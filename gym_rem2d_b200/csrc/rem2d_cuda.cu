// rem2d_cuda.cu — host side + C-ABI (include/rem2d.h, include/rem2d_stats.h, include/rem2d_control.h, include/rem2d_policy.h) of the CUDA build, sm_100a only (kernels: rem2d_kernels.cu).
//
// Sorts creatures into capacity classes (by body count), keeps one lane-interleaved state block per 32 creatures in
// HBM, and runs every class on its own stream so small and large classes overlap on the 148 SMs: rem2d_step on a
// static creature -> lane mapping, rem2d_run_episodes / rem2d_evaluate on persistent warps that pull creatures from a
// per-class queue (bulk mode), hand long-lived creatures to warp-per-creature launches (tail mode), or give every
// creature its own warp when the population is small. There is no CPU physics fallback: every tick is computed by
// rem2d::Sim::tick on the device.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <thread>
#include <string>
#include <vector>

#include "rem2d_classes.h"
#include "rem2d_host_util.h"
#include "../../include/rem2d_control.h"
#include "../../include/rem2d_policy.h"

using namespace rem2d;

// capacity class k (rem2d_host_util.h: class_dims)
static ClassOps g_classes(int k) { return ClassOps(class_dims[k].nb, class_dims[k].nc, class_dims[k].nt); }

// fitness / ticks / alive / status of every creature of a class -> creature-indexed outputs
__global__ void gather_kernel(const float* state, const int* __restrict__ lane_creature, int n_lanes, int words,
                              double* fitness, int* ticks, int* alive, int* status) {
    int gl = blockIdx.x * blockDim.x + threadIdx.x;
    if (gl >= n_lanes) return;
    int c = lane_creature[gl];
    if (c < 0) return;
    const float* g = state + (size_t)(gl >> 5) * words * 32 + (gl & 31);
    fitness[c] = __hiloint2double(__float_as_int(g[S_FIT_HI * 32]), __float_as_int(g[S_FIT_LO * 32]));
    ticks[c] = __float_as_int(g[S_TICKS * 32]);
    alive[c] = __float_as_int(g[S_ALIVE * 32]);
    status[c] = __float_as_int(g[S_STATUS * 32]);
}

// root x / wall of death / alive of every creature of a class -> creature-indexed outputs (rem2d_read_roots)
__global__ void roots_kernel(const float* state, const int* __restrict__ lane_creature, int n_lanes, int words,
                             float* root_x, double* wod, int* alive) {
    int gl = blockIdx.x * blockDim.x + threadIdx.x;
    if (gl >= n_lanes) return;
    int c = lane_creature[gl];
    if (c < 0) return;
    const float* g = state + (size_t)(gl >> 5) * words * 32 + (gl & 31);
    root_x[c] = g[(S_COUNT + BF_CX) * 32];
    wod[c] = __hiloint2double(__float_as_int(g[S_WOD_HI * 32]), __float_as_int(g[S_WOD_LO * 32]));
    alive[c] = __float_as_int(g[S_ALIVE * 32]);
}

// joint angles / joint speeds / root state / ground flags of every creature of a class -> table-indexed outputs
// (rem2d_read_observations; rem2d::observe_column)
__global__ void observations_kernel(const float* state, const int* __restrict__ lane_creature, int n_lanes, const __grid_constant__ Layout L,
                                    const int32_t* __restrict__ body_off, float* joint_angle, float* joint_speed, float* root, int32_t* ground) {
    int gl = blockIdx.x * blockDim.x + threadIdx.x;
    if (gl >= n_lanes) return;
    int c = lane_creature[gl];
    if (c < 0) return;
    const float* g = state + (size_t)(gl >> 5) * L.words * 32 + (gl & 31);
    const int b0 = body_off[c], j0 = b0 - c;
    observe_column(g, L, body_off[c + 1] - b0, joint_angle + j0, joint_speed + j0, root + (size_t)c * 6, ground + b0);
}

// FP32 issue-rate microbenchmark: 8 independent multiply / add chains per thread. The step kernel is built with
// -fmad=false (parity), so its ceiling is the non-fused FMUL/FADD issue rate: 1 FLOP per lane per cycle.
__global__ void fp32_issue_kernel(float* out, int iters, float b, float c) {
    float a0 = threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    for (int i = 0; i < iters; ++i) {
        a0 = a0 * b; a1 = a1 * b; a2 = a2 * b; a3 = a3 * b; a4 = a4 * b; a5 = a5 * b; a6 = a6 * b; a7 = a7 * b;
        a0 = a0 + c; a1 = a1 + c; a2 = a2 + c; a3 = a3 + c; a4 = a4 + c; a5 = a5 + c; a6 = a6 + c; a7 = a7 + c;
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// ------------------------------------------------------------------ handle
// Device buffers are grow-only and reused across uploads: re-allocating ~1 GB of state blocks on every rem2d_evaluate
// call cost ~0.4 s per generation.
#define N_COUNTER_WORDS (REM2D_N_COUNTERS + 12 * 16)      // work counters + phase cycles of diagnostic builds (REM2D_PHASE_TIMING)
struct Buf { void* p = nullptr; size_t cap = 0; };
static cudaError_t ensure(Buf& b, size_t bytes) {
    if (bytes <= b.cap && b.p) return cudaSuccess;
    // a buffer that has to grow will grow again (an evolving population shifts towards the large classes generation by
    // generation): 50 % headroom then, 12.5 % on the first allocation
    const bool regrow = b.p != nullptr;
    if (b.p) cudaFree(b.p);
    b.p = nullptr; b.cap = 0;
    size_t want = bytes + (regrow ? bytes / 2 : bytes / 8) + 256;
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e == cudaSuccess) b.cap = want;
    return e;
}

struct ClassState {
    std::vector<int> lane_creature;     // host copy: [n_batches*32], -1 = padding lane
    int n_batches = 0;
    int n_members = 0;                  // creatures of this class (lane_creature[0..n_members) are real)
    cudaStream_t stream2 = nullptr;     // overflow wave
    cudaEvent_t done2 = nullptr;
    float* d_state = nullptr;
    int* d_lane_creature = nullptr;
    int* d_queue = nullptr;
    float* d_park_state = nullptr;      // columns of the parked creatures, by park slot
    int* d_park_creature = nullptr;     // park slot -> creature + 1 (0: allocated, not yet published)
    int* d_park_count = nullptr;        // park slots handed out
    int* h_park_count = nullptr;        // pinned, see launch_episodes
    Buf b_state, b_park_state, b_lc, b_park_creature, b_small, b_trace, b_ttrace;   // backing storage (grow-only)
    Buf b_redo_order, b_redo_slots;     // promotion re-runs (grow-only)
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    cudaEvent_t t_begin = nullptr, t_end = nullptr;     // per-class timeline of the last rem2d_run_episodes (diagnostics)
};

struct rem2d_handle {
    rem2d_config cfg;
    Options opt;
    PlanInput load;                     // device and class sizes of the uploaded population, as the planner sees them
    UploadPlan plan{};                  // group widths, grids and kernel image of the uploaded population (plan_upload)
    cudaStream_t user_stream = nullptr;
    Terrain* d_ter = nullptr;
    Consts* d_consts = nullptr;
    unsigned long long* d_counters = nullptr;
    // Tail-mode launches are made on demand, each on a stream of this pool that is idle at that moment: a tail launch lives as
    // long as its longest creature (hundreds of ms), so a second kernel queued behind it on the same stream would wait for
    // it (and block its hardware queue for other streams). The pool grows when no stream is idle.
    std::vector<cudaStream_t> tail_pool;
    std::vector<char> tail_used;         // streams that received work during the current rem2d_run_episodes
    cudaStream_t poll_stream = nullptr;
    cudaEvent_t pool_done = nullptr;
    int* h_poll = nullptr;               // pinned [N_CLASSES]
    bool have_terrain = false, have_pop = false;
    bool state_valid = false;           // per-creature state blocks hold a consistent snapshot (reset/step path)
    bool results_valid = false;         // d_fitness/d_ticks/... were written by the episode kernel
    // episode statistics (rem2d_set_stats): the flag, its value at the upload (selects the statistics images for the runs of
    // that upload), and whether the statistics buffers hold those of the last run
    bool stats_on = false, upload_stats = false, stats_valid = false;
    Buf b_stats;
    EpisodeStats dstats{};
    // feedback policy (rem2d_set_policy): the caller's weights for later uploads, and the snapshot the current upload took on
    // the device (selects the policy images for every run of that upload; the statistics then always point somewhere, b_stats)
    std::vector<double> policy_w;
    int policy_nj = 0, policy_hidden = 0;
    bool policy_on = false, upload_policy = false;
    Buf b_policy;
    PolicyWeights dpolicy{};
    int warps_per_sm[6] = {};           // rem2d_episode_blocks_per_sm of the six episode images (plan_upload input)
    int prio_high = 0;                  // greatest stream priority of the device (tail pool)
    int n_edges = 0;
    // population
    int n_creatures = 0, n_bodies = 0, n_joints = 0;
    std::vector<int32_t> body_off;
    std::vector<float> priority;         // rem2d_set_priority: expected lifetimes for the next upload (empty: none)
    std::vector<int> creature_class, creature_lane;     // lane index within the class (batch*32+lane)
    Buf d_pop_mem[16];
    Buf b_results, b_roots;
    Buf b_targets, b_obs;               // rem2d_step_targets / rem2d_read_observations (grow-only)
    DevPop dpop{};
    ClassState cls[N_CLASSES];
    double* d_fitness = nullptr; int *d_ticks = nullptr, *d_alive = nullptr, *d_status = nullptr;
    std::vector<double> h_fitness; std::vector<int> h_ticks, h_alive, h_status;
    cudaEvent_t ev_start = nullptr, ev_stop = nullptr, ev_fork = nullptr;
    float last_ms = 0.0f;
    int64_t launches = 0;
    std::string err;
};

static thread_local std::string g_create_err;



#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e_);                                 \
            return REM2D_E_CUDA;                                                                         \
        }                                                                                                \
    } while (0)

static bool set_option(Options& o, const char* name, double v) {
    const std::string n(name);
    if (n == "warp_mode_max") o.warp_mode_max = (int)v;
    else if (n == "park_ticks") o.park_ticks = (int)v;
    else if (n == "park_cap") o.park_cap = v;
    else if (n == "smem_budget_kb") o.smem_budget_kb = v;
    else if (n == "group_shift") o.group_shift = (int)v;
    else if (n == "tail_group_shift") o.tail_group_shift = std::max(0, std::min(5, (int)v));
    else if (n == "trace") o.trace = (int)v;
    else if (n == "image") o.image = std::max(-1, std::min(1, (int)v));
    else if (n == "overflow_wave") o.overflow_wave = (int)v != 0;
    else if (n.rfind("class_gs_", 0) == 0 && n.size() == 10 && n[9] >= '0' && n[9] < '0' + N_CLASSES) o.class_gs[n[9] - '0'] = (int)v;
    else return false;
    return true;
}
static void options_from_env(Options& o) {
    static const char* names[] = {"warp_mode_max", "park_ticks", "park_cap", "smem_budget_kb",
                                  "group_shift", "tail_group_shift", "trace", "image", "overflow_wave"};
    for (const char* n : names) {
        std::string env = "REM2D_";
        for (const char* q = n; *q; ++q) env += (char)toupper(*q);
        if (const char* e = getenv(env.c_str())) set_option(o, n, atof(e));
    }
    if (const char* e = getenv("REM2D_CLASS_GS"))          // "0,0,1,2,2,2,2,3,3": group shift per capacity class
        for (int k = 0; k < N_CLASSES && *e; ++k) { o.class_gs[k] = atoi(e); while (*e && *e != ',') ++e; if (*e == ',') ++e; }
}

static void free_population(rem2d_handle* h) {          // logical reset; the buffers stay allocated for reuse
    for (auto& c : h->cls) { c.n_batches = 0; c.n_members = 0; c.lane_creature.clear(); }
    h->have_pop = false; h->state_valid = false; h->results_valid = false; h->stats_valid = false;
}
static void release_buffers(rem2d_handle* h) {
    for (auto& b : h->d_pop_mem) { if (b.p) cudaFree(b.p); b = Buf(); }
    for (auto& c : h->cls) {
        Buf* bufs[] = {&c.b_state, &c.b_park_state, &c.b_lc, &c.b_park_creature, &c.b_small, &c.b_trace, &c.b_ttrace,
                       &c.b_redo_order, &c.b_redo_slots};
        for (Buf* b : bufs) { if (b->p) cudaFree(b->p); *b = Buf(); }
        if (c.h_park_count) cudaFreeHost(c.h_park_count);
        c.h_park_count = nullptr;
    }
    if (h->b_results.p) cudaFree(h->b_results.p);
    h->b_results = Buf();
    if (h->b_roots.p) cudaFree(h->b_roots.p);
    h->b_roots = Buf();
    if (h->b_stats.p) cudaFree(h->b_stats.p);
    h->b_stats = Buf();
    for (Buf* b : {&h->b_targets, &h->b_obs, &h->b_policy}) { if (b->p) cudaFree(b->p); *b = Buf(); }
}

extern "C" {

void rem2d_default_config(rem2d_config* cfg) {
    memset(cfg, 0, sizeof(*cfg));
    cfg->dt = (float)(1.0 / 50);        // Modular2DEnv.py:26,634
    cfg->velocity_iterations = 180;     // Modular2DEnv.py:634
    cfg->position_iterations = 60;
    cfg->gravity_y = -10.0f;
    cfg->module_friction = (float)0.1;  // simple_module.py:289
    cfg->terrain_friction = 2.5f;       // Modular2DEnv.py:62
    cfg->p_gain = 1.9;                  // Modular2DEnv.py:601
    cfg->wod_speed = 0.04;              // Modular2DEnv.py:52
    cfg->env_length = 100.0;            // REM2D_main.py:350
    cfg->evaluation_steps = 10000;      // REM2D_main.py:350
    cfg->continuous = 1;
    cfg->allow_sleep = 1;
    cfg->terminate = 1;
    cfg->device = 0;
    cfg->stream = nullptr;
    cfg->sincos_mode = 0;
}
int rem2d_abi_version(void) { return REM2D_ABI_VERSION; }
const char* rem2d_backend(void) { return "cuda-sm_100a"; }

int rem2d_create(const rem2d_config* cfg, rem2d_handle** out) {
    if (!cfg || !out) { g_create_err = "rem2d_create: NULL argument"; return REM2D_E_INVALID; }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_create_err = std::string("rem2d_create: no CUDA device (") + cudaGetErrorString(e) + "); this library has no CPU fallback";
        return REM2D_E_CUDA;
    }
    if (cfg->device < 0 || cfg->device >= ndev) { g_create_err = "rem2d_create: bad device ordinal"; return REM2D_E_INVALID; }
    if (cfg->sincos_mode != 0) { g_create_err = "rem2d_create: sincos_mode != 0 is an oracle-only option"; return REM2D_E_INVALID; }
    e = cudaSetDevice(cfg->device);
    if (e != cudaSuccess) { g_create_err = std::string("cudaSetDevice: ") + cudaGetErrorString(e); return REM2D_E_CUDA; }
    rem2d_handle* h = new rem2d_handle();
    h->cfg = *cfg;
    h->user_stream = (cudaStream_t)cfg->stream;
    options_from_env(h->opt);
    // every failure path releases what was created so far (rem2d_destroy copes with a partially built handle)
    auto fail = [&](const char* what, cudaError_t err) { g_create_err = std::string(what) + ": " + cudaGetErrorString(err); rem2d_destroy(h); return REM2D_E_CUDA; };
    if ((e = cudaMalloc(&h->d_ter, sizeof(Terrain))) != cudaSuccess) return fail("cudaMalloc terrain", e);
    if ((e = cudaMalloc(&h->d_consts, sizeof(Consts))) != cudaSuccess) return fail("cudaMalloc consts", e);
    if ((e = cudaMalloc(&h->d_counters, sizeof(unsigned long long) * N_COUNTER_WORDS)) != cudaSuccess) return fail("cudaMalloc counters", e);
    if ((e = cudaMemset(h->d_counters, 0, sizeof(unsigned long long) * N_COUNTER_WORDS)) != cudaSuccess) return fail("cudaMemset counters", e);
    Consts k = make_consts(cfg);
    if ((e = cudaMemcpy(h->d_consts, &k, sizeof(k), cudaMemcpyHostToDevice)) != cudaSuccess) return fail("cudaMemcpy consts", e);
    for (auto& c : h->cls) {
        if ((e = cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking)) != cudaSuccess) return fail("cudaStreamCreate", e);
        if ((e = cudaStreamCreateWithFlags(&c.stream2, cudaStreamNonBlocking)) != cudaSuccess) return fail("cudaStreamCreate", e);
        if ((e = cudaEventCreateWithFlags(&c.done2, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
        if ((e = cudaEventCreateWithFlags(&c.done, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
        if ((e = cudaEventCreate(&c.t_begin)) != cudaSuccess || (e = cudaEventCreate(&c.t_end)) != cudaSuccess) return fail("cudaEventCreate", e);
    }
    if ((e = cudaEventCreate(&h->ev_start)) != cudaSuccess || (e = cudaEventCreate(&h->ev_stop)) != cudaSuccess) return fail("cudaEventCreate", e);
    {   // tail launches and the polling copies run at the device's greatest stream priority: their CTAs / copies go ahead of
        // the queued overflow-wave CTAs of the episode launches
        int least = 0, greatest = 0;
        if (cudaDeviceGetStreamPriorityRange(&least, &greatest) == cudaSuccess) h->prio_high = greatest;
        else cudaGetLastError();
    }
    h->tail_pool.assign(64, nullptr);
    for (auto& st : h->tail_pool)
        if ((e = cudaStreamCreateWithPriority(&st, cudaStreamNonBlocking, h->prio_high)) != cudaSuccess) return fail("cudaStreamCreate (tail pool)", e);
    if ((e = cudaStreamCreateWithPriority(&h->poll_stream, cudaStreamNonBlocking, h->prio_high)) != cudaSuccess) return fail("cudaStreamCreate (poll)", e);
    if ((e = cudaEventCreateWithFlags(&h->pool_done, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
    if ((e = cudaMallocHost(&h->h_poll, sizeof(int) * 16)) != cudaSuccess) return fail("cudaMallocHost", e);
    if ((e = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
    cudaDeviceGetAttribute(&h->load.n_sms, cudaDevAttrMultiProcessorCount, cfg->device);
    {
        int max_hot = 0;
        for (int q = 0; q < N_CLASSES; ++q)
            for (int gs = 0; gs <= 5; ++gs) max_hot = std::max(max_hot, class_hot_bytes(q, gs));
        if ((e = rem2d_set_kernel_attributes(max_hot)) != cudaSuccess) return fail("cudaFuncSetAttribute", e);
        for (int im = 0; im < 6; ++im) h->warps_per_sm[im] = std::max(1, rem2d_episode_blocks_per_sm(im, 1024));
        for (int im = 0; im < 2; ++im) h->load.max_warps_per_sm[im] = h->warps_per_sm[im];
    }
    *out = h;
    return REM2D_OK;
}

int rem2d_set_option(rem2d_handle* h, const char* name, double value) {
    if (!h || !name) return REM2D_E_INVALID;
    if (!set_option(h->opt, name, value)) { h->err = std::string("set_option: unknown option ") + name; return REM2D_E_INVALID; }
    return REM2D_OK;
}

int rem2d_destroy(rem2d_handle* h) {
    if (!h) return REM2D_E_INVALID;
    cudaSetDevice(h->cfg.device);
    cudaDeviceSynchronize();
    free_population(h);
    release_buffers(h);
    for (auto& c : h->cls) {
        if (c.stream) cudaStreamDestroy(c.stream);
        if (c.stream2) cudaStreamDestroy(c.stream2);
        if (c.done) cudaEventDestroy(c.done);
        if (c.done2) cudaEventDestroy(c.done2);
        if (c.t_begin) cudaEventDestroy(c.t_begin);
        if (c.t_end) cudaEventDestroy(c.t_end);
    }
    for (auto& st : h->tail_pool) if (st) cudaStreamDestroy(st);
    if (h->poll_stream) cudaStreamDestroy(h->poll_stream);
    if (h->pool_done) cudaEventDestroy(h->pool_done);
    if (h->h_poll) cudaFreeHost(h->h_poll);
    if (h->ev_start) cudaEventDestroy(h->ev_start);
    if (h->ev_stop) cudaEventDestroy(h->ev_stop);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->d_ter) cudaFree(h->d_ter);
    if (h->d_consts) cudaFree(h->d_consts);
    if (h->d_counters) cudaFree(h->d_counters);
    cudaGetLastError();
    delete h;
    return REM2D_OK;
}

const char* rem2d_last_error(rem2d_handle* h) { return h ? h->err.c_str() : g_create_err.c_str(); }

int rem2d_set_terrain(rem2d_handle* h, const double* y, int32_t n, double step) {
    if (!h) return REM2D_E_INVALID;
    if (!y || n < 2 || n > RB_MAX_EDGES) { h->err = "set_terrain: need 2..200 vertices"; return REM2D_E_INVALID; }
    cudaSetDevice(h->cfg.device);
    Terrain* t = new Terrain();
    fill_terrain(t, y, n, step);
    cudaError_t e = cudaMemcpy(h->d_ter, t, sizeof(Terrain), cudaMemcpyHostToDevice);
    delete t;
    if (e != cudaSuccess) { h->err = std::string("set_terrain: ") + cudaGetErrorString(e); return REM2D_E_CUDA; }
    h->n_edges = n - 1;
    h->have_terrain = true;
    return REM2D_OK;
}

}  // extern "C"

template <typename T>
static cudaError_t upload_array(rem2d_handle* h, int slot, const T* src, size_t n, const T** dst) {
    cudaError_t e = ensure(h->d_pop_mem[slot], (n ? n : 1) * sizeof(T));
    if (e != cudaSuccess) return e;
    void* d = h->d_pop_mem[slot].p;
    if (n) e = cudaMemcpyAsync(d, src, n * sizeof(T), cudaMemcpyHostToDevice, h->user_stream);
    *dst = (const T*)d;
    return e;
}

static int launch_reset(rem2d_handle* h);

static int upload_impl(rem2d_handle* h, const rem2d_population* pop, bool do_reset) {
    if (!h || !pop) return REM2D_E_INVALID;
    if (pop->n_creatures < 0 || pop->n_joints != pop->n_bodies - pop->n_creatures) { h->err = "upload: inconsistent counts"; return REM2D_E_INVALID; }
    if (h->policy_on && pop->n_joints != h->policy_nj) {
        h->err = "upload: the policy set with rem2d_set_policy has " + std::to_string(h->policy_nj) + " joints, the population " +
                 std::to_string(pop->n_joints);
        return REM2D_E_INVALID;
    }
    cudaSetDevice(h->cfg.device);
    free_population(h);
    const int n = pop->n_creatures;
    h->n_creatures = n; h->n_bodies = pop->n_bodies; h->n_joints = pop->n_joints;
    h->body_off.assign(pop->body_off, pop->body_off + n + 1);
    // classify + validate
    h->creature_class.assign(n, -1);
    h->creature_lane.assign(n, -1);
    std::vector<std::vector<int>> members(N_CLASSES);
    for (int c = 0; c < n; ++c) {
        int nb = pop->body_off[c + 1] - pop->body_off[c];
        if (nb < 1) { h->err = "upload: creature without a root body"; return REM2D_E_INVALID; }
        int k = -1;
        for (int q = 0; q < N_CLASSES; ++q) if (nb <= class_dims[q].nb) { k = q; break; }
        if (k < 0) { char buf[128]; snprintf(buf, sizeof(buf), "upload: creature %d has %d bodies (> %d supported)", c, nb, class_dims[N_CLASSES - 1].nb); h->err = buf; return REM2D_E_CAPACITY; }
        int j0 = pop->body_off[c] - c;
        for (int j = 0; j < nb - 1; ++j)
            if (pop->joint_parent[j0 + j] < 0 || pop->joint_parent[j0 + j] > j) { h->err = "upload: joint parent must precede its child"; return REM2D_E_INVALID; }
        h->creature_class[c] = k;
        members[k].push_back(c);
    }
    std::vector<uint8_t> order((size_t)std::max(pop->n_joints, 1), 0);
    for (int c = 0; c < n; ++c) {
        int nb = pop->body_off[c + 1] - pop->body_off[c], j0 = pop->body_off[c] - c;
        island_joint_order(nb, pop->joint_parent + j0, order.data() + j0);
    }
    size_t nbod = (size_t)pop->n_bodies, nj = (size_t)pop->n_joints;
    CK(upload_array(h, 0, pop->body_off, (size_t)n + 1, &h->dpop.body_off));
    CK(upload_array(h, 1, pop->shape, nbod, &h->dpop.shape));
    CK(upload_array(h, 2, pop->hx, nbod, &h->dpop.hx));
    CK(upload_array(h, 3, pop->hy, nbod, &h->dpop.hy));
    CK(upload_array(h, 4, pop->x0, nbod, &h->dpop.x0));
    CK(upload_array(h, 5, pop->y0, nbod, &h->dpop.y0));
    CK(upload_array(h, 6, pop->a0, nbod, &h->dpop.a0));
    CK(upload_array(h, 7, pop->joint_parent, nj, &h->dpop.joint_parent));
    CK(upload_array(h, 8, pop->anchor_a, nj * 2, &h->dpop.anchor_a));
    CK(upload_array(h, 9, pop->anchor_b, nj * 2, &h->dpop.anchor_b));
    CK(upload_array(h, 10, pop->lower, nj, &h->dpop.lower));
    CK(upload_array(h, 11, pop->upper, nj, &h->dpop.upper));
    CK(upload_array(h, 12, pop->max_torque, nj, &h->dpop.max_torque));
    CK(upload_array(h, 13, pop->ctrl, nbod * 5, &h->dpop.ctrl));
    CK(upload_array(h, 14, (const uint8_t*)order.data(), nj, &h->dpop.joint_order));
    // the policy's snapshot (rem2d_set_policy): later calls change h->policy_w, never this copy
    h->upload_policy = h->policy_on;
    if (h->upload_policy) {
        CK(ensure(h->b_policy, sizeof(double) * std::max<size_t>(h->policy_w.size(), 1)));
        if (!h->policy_w.empty())
            CK(cudaMemcpyAsync(h->b_policy.p, h->policy_w.data(), sizeof(double) * h->policy_w.size(), cudaMemcpyHostToDevice, h->user_stream));
        h->dpolicy = PolicyWeights{(const double*)h->b_policy.p, h->dpop.body_off, h->policy_hidden};
    }
    // the pageable source buffers (order, caller arrays) must stay valid until the copies ran
    CK(cudaStreamSynchronize(h->user_stream));
    for (int k = 0; k < N_CLASSES; ++k) {
        auto& m = members[k];
        if (m.empty()) continue;
        // big creatures first: batches of similar size limit lane divergence, and the costly batches start early; creatures
        // the caller expects to be long-lived (rem2d_set_priority: >= 130 ticks, i.e. they outrun the wall of death) go to
        // the very front of the class queue, the longest-lived first in buckets of 32 ticks (longest-processing-time-first).
        // Measured with the parents' lifetimes as the hint (profiles/r2_ea_pop_sweep.txt): selected populations, where most
        // creatures are long-lived, evaluate 7-11 % faster with the ordering than with the threshold alone (1570 -> 1480,
        // 2575 -> 2380, 2130 -> 1900 ms); a random population with a perfect hint gains 20 % either way (800 -> 640 ms).
        const bool prio = (int)h->priority.size() == n;
        // "long-lived" = expected to be alive when the wall of death has passed the start pad (root at x = 5: tick 125 at the
        // reference's 0.04 per tick, + 4 %)
        const float long_lived = (h->cfg.terminate && h->cfg.wod_speed > 0.0) ? (float)(5.2 / h->cfg.wod_speed) : 130.0f;
        std::stable_sort(m.begin(), m.end(), [&](int a, int b) {
            int la = prio && h->priority[a] >= long_lived, lb = prio && h->priority[b] >= long_lived;
            if (prio) {      // ... and among those the longest expected lifetime first, in buckets of 32 ticks
                la = la ? 1 + ((int)std::min(h->priority[a], 8192.0f) >> 5) : 0;
                lb = lb ? 1 + ((int)std::min(h->priority[b], 8192.0f) >> 5) : 0;
            }
            if (la != lb) return la > lb;
            return (pop->body_off[a + 1] - pop->body_off[a]) > (pop->body_off[b + 1] - pop->body_off[b]);
        });
        ClassState& cs = h->cls[k];
        cs.n_batches = (int)((m.size() + 31) / 32);
        cs.n_members = (int)m.size();
        cs.lane_creature.assign((size_t)cs.n_batches * 32, -1);
        for (size_t i = 0; i < m.size(); ++i) { cs.lane_creature[i] = m[i]; h->creature_lane[m[i]] = (int)i; }
        const size_t lane_bytes = cs.lane_creature.size() * sizeof(int);
        // (+2: the overflow wave's columns start at the block after the first launch's and end on a whole group)
        const size_t state_bytes = (size_t)(cs.n_batches + 2) * g_classes(k).words * 32 * sizeof(float);
        CK(ensure(cs.b_lc, lane_bytes)); cs.d_lane_creature = (int*)cs.b_lc.p;
        CK(cudaMemcpy(cs.d_lane_creature, cs.lane_creature.data(), cs.lane_creature.size() * sizeof(int), cudaMemcpyHostToDevice));
        CK(ensure(cs.b_state, state_bytes)); cs.d_state = (float*)cs.b_state.p;
        CK(ensure(cs.b_park_state, state_bytes)); cs.d_park_state = (float*)cs.b_park_state.p;
        CK(ensure(cs.b_park_creature, lane_bytes)); cs.d_park_creature = (int*)cs.b_park_creature.p;
        CK(ensure(cs.b_small, 64)); cs.d_park_count = (int*)cs.b_small.p; cs.d_queue = (int*)cs.b_small.p + 4;
        if (!cs.h_park_count) CK(cudaMallocHost(&cs.h_park_count, sizeof(int)));
    }
    // per-creature cost ~ tick latency of its size: measured ~0.3 ms + 0.085 ms per body for a resident warp; lone bodies
    // fall asleep after landing and cost almost nothing
    for (int k = 0; k < N_CLASSES; ++k) {
        h->load.members[k] = h->cls[k].n_members;
        h->load.work[k] = 0.0;
        for (int c : members[k]) { int nbc = pop->body_off[c + 1] - pop->body_off[c]; h->load.work[k] += nbc == 1 ? 1.0 : 3.5 + nbc; }
    }
    // statistics runs launch the statistics images, policy runs the policy images: the planner sees their occupancy
    h->upload_stats = h->stats_on;
    for (int im = 0; im < 2; ++im) h->load.max_warps_per_sm[im] = h->warps_per_sm[im + (h->upload_policy ? 4 : h->upload_stats ? 2 : 0)];
    h->plan = plan_upload(h->load, h->opt);
    if (h->upload_stats || h->upload_policy) {      // (the policy images always accumulate: without statistics into scratch)
        const size_t nn = (size_t)std::max(n, 1), nbod = (size_t)std::max(pop->n_bodies, 1);
        CK(ensure(h->b_stats, nn * (sizeof(double) + sizeof(float) + 2 * sizeof(int32_t)) + nbod * sizeof(int32_t) + 64));
        EpisodeStats& d = h->dstats;
        d.joint_work = (double*)h->b_stats.p;
        d.max_x = (float*)(d.joint_work + nn);
        d.end_reason = (int32_t*)(d.max_x + nn);
        d.airborne_ticks = d.end_reason + nn;
        d.ground_ticks = d.airborne_ticks + nn;
        d.body_off = h->dpop.body_off;
    }
    {
        const size_t nn = (size_t)std::max(n, 1);
        CK(ensure(h->b_results, nn * (sizeof(double) + 3 * sizeof(int))));
        h->d_fitness = (double*)h->b_results.p;
        h->d_ticks = (int*)(h->d_fitness + nn);
        h->d_alive = h->d_ticks + nn;
        h->d_status = h->d_alive + nn;
    }
    h->h_fitness.assign(n, 0.0); h->h_ticks.assign(n, 0); h->h_alive.assign(n, 0); h->h_status.assign(n, 0);
    h->have_pop = true;
    h->priority.clear();                 // the hint applies to one upload
    return do_reset ? launch_reset(h) : REM2D_OK;
}

extern "C" int rem2d_upload(rem2d_handle* h, const rem2d_population* pop) { return upload_impl(h, pop, true); }

// fork the class streams off the user stream / join them back
static int fork_streams(rem2d_handle* h) {
    CK(cudaEventRecord(h->ev_fork, h->user_stream));
    for (auto& c : h->cls) if (c.n_batches) { CK(cudaStreamWaitEvent(c.stream, h->ev_fork, 0)); CK(cudaStreamWaitEvent(c.stream2, h->ev_fork, 0)); }
    return REM2D_OK;
}
static int join_streams(rem2d_handle* h) {
    for (auto& c : h->cls) if (c.n_batches) {
        CK(cudaEventRecord(c.done, c.stream)); CK(cudaStreamWaitEvent(h->user_stream, c.done, 0));
        CK(cudaEventRecord(c.done2, c.stream2)); CK(cudaStreamWaitEvent(h->user_stream, c.done2, 0));
    }
    return REM2D_OK;
}

static int launch_reset(rem2d_handle* h) {
    if (!h->have_terrain) { h->err = "reset: no terrain set"; return REM2D_E_INVALID; }
    int rc = fork_streams(h);
    if (rc) return rc;
    for (int k = N_CLASSES - 1; k >= 0; --k) {
        ClassState& cs = h->cls[k];
        if (!cs.n_batches) continue;
        g_classes(k).reset(step_group_shift(h->load, k, h->opt), cs.n_batches, cs.stream, cs.d_state, cs.d_lane_creature, h->dpop);
        h->launches++;
    }
    CK(cudaGetLastError());
    rc = join_streams(h);
    if (rc) return rc;
    CK(cudaMemsetAsync(h->d_counters, 0, sizeof(unsigned long long) * N_COUNTER_WORDS, h->user_stream));
    h->state_valid = true; h->results_valid = false; h->stats_valid = false;
    return REM2D_OK;
}

// Promotion: creatures that exceeded a capacity of their class (contact pool) are re-run from tick 0 on the refill
// episode kernel of the next larger class until they fit. Rare (very fine terrains, pile-ups).
// destinations of the episode statistics of the uploaded population (nullptr: it was uploaded with statistics off and without a
// policy; the policy images accumulate them anyway, into b_stats, which read_stats then refuses)
static const EpisodeStats* stats_dest(const rem2d_handle* h) { return h->upload_stats || h->upload_policy ? &h->dstats : nullptr; }
// the policy of the uploaded population (nullptr: none)
static const PolicyWeights* policy_of(const rem2d_handle* h) { return h->upload_policy ? &h->dpolicy : nullptr; }

static int promote_overflowed(rem2d_handle* h, int max_ticks) {
    const int n = h->n_creatures;
    std::vector<int> cls_of(h->creature_class);
    for (int round = 0; round < N_CLASSES; ++round) {
        CK(cudaMemcpyAsync(h->h_status.data(), h->d_status, sizeof(int) * n, cudaMemcpyDeviceToHost, h->user_stream));
        CK(cudaStreamSynchronize(h->user_stream));
        std::vector<std::vector<int>> redo(N_CLASSES);
        bool any = false;
        for (int c = 0; c < n; ++c)
            if (h->h_status[c]) {
                if (cls_of[c] + 1 >= N_CLASSES) {
                    char buf[160];
                    snprintf(buf, sizeof(buf), "creature %d exceeds the capacities of the largest class (status %d)", c, h->h_status[c]);
                    h->err = buf;
                    return REM2D_E_CAPACITY;
                }
                cls_of[c] += 1;
                redo[cls_of[c]].push_back(c);
                any = true;
            }
        if (!any) break;
        for (int k = 0; k < N_CLASSES; ++k) {
            if (redo[k].empty()) continue;
            ClassState& cs = h->cls[k];
            const int gs = h->plan.gs[k], per = 32 >> gs;
            const int grid = (int)((redo[k].size() + per - 1) / per), batches = (int)((redo[k].size() + 31) / 32);
            CK(ensure(cs.b_redo_order, sizeof(int) * (redo[k].size() + 1)));
            CK(ensure(cs.b_redo_slots, (size_t)batches * g_classes(k).words * 32 * sizeof(float)));
            int* d_order = (int*)cs.b_redo_order.p;
            int* d_queue = d_order + redo[k].size();
            CK(cudaMemcpyAsync(d_order, redo[k].data(), sizeof(int) * redo[k].size(), cudaMemcpyHostToDevice, h->user_stream));
            CK(cudaMemsetAsync(d_queue, 0, sizeof(int), h->user_stream));
            g_classes(k).episode(h->plan.image, gs, widest_group_shift(k, gs), grid, h->user_stream, (float*)cs.b_redo_slots.p, d_order, (int)redo[k].size(), d_queue, h->dpop, h->d_ter,
                                 h->d_consts, max_ticks, h->d_fitness, h->d_ticks, h->d_alive, h->d_status, h->d_counters,
                                 ParkPolicy{0, 0, 0.0f, 0, 0, 0, nullptr, nullptr, 0}, nullptr, nullptr, nullptr, stats_dest(h), policy_of(h));
            h->launches++;
            CK(cudaGetLastError());
            CK(cudaStreamSynchronize(h->user_stream));      // redo[] (pageable source of the copy) goes out of scope
        }
    }
    return REM2D_OK;
}

// Whole episodes for the uploaded population on the persistent episode kernels (one per class, concurrent).
static int launch_episodes(rem2d_handle* h, int max_ticks) {
    if (!h->have_terrain) { h->err = "run_episodes: no terrain set"; return REM2D_E_INVALID; }
    h->stats_valid = false;
    const LaunchPlan lp = plan_launch(h->load, h->plan, max_ticks, h->opt);
    const bool trace = h->opt.trace != 0;
    auto park_policy = [&](int k) {
        return ParkPolicy{lp.park_ticks, lp.park_cap[k], 0.0f, 0, h->cls[k].n_members, lp.park_ticks, nullptr,
                          trace ? (unsigned int*)h->cls[k].b_ttrace.p : nullptr, h->opt.tail_group_shift};
    };
    CK(cudaMemsetAsync(h->d_counters, 0, sizeof(unsigned long long) * N_COUNTER_WORDS, h->user_stream));
    CK(cudaEventRecord(h->ev_start, h->user_stream));
    int rc = fork_streams(h);
    if (rc) return rc;
    for (int oi = 0; oi < N_CLASSES; ++oi) {
        const int k = lp.order[oi];
        ClassState& cs = h->cls[k];
        if (!cs.n_batches) continue;
        CK(cudaMemsetAsync(cs.d_queue, 0, sizeof(int), cs.stream));
        CK(cudaEventRecord(cs.t_begin, cs.stream));
        if (lp.warp_mode) {      // queue mode with a whole warp per creature and one warp for every creature
            g_classes(k).episode(1, 5, 5, cs.n_members, cs.stream, cs.d_state, cs.d_lane_creature, cs.n_members, cs.d_queue, h->dpop, h->d_ter,
                                 h->d_consts, max_ticks, h->d_fitness, h->d_ticks, h->d_alive, h->d_status, h->d_counters,
                                 ParkPolicy{0, 0, 0.0f, 0, 0, 0, nullptr, nullptr, 0}, nullptr, nullptr, nullptr, stats_dest(h), policy_of(h));
            CK(cudaEventRecord(cs.t_end, cs.stream));
            h->launches++;
            continue;
        }
        CK(cudaMemsetAsync(cs.d_park_count, 0, sizeof(int), cs.stream));
        CK(cudaMemsetAsync(cs.d_park_creature, 0, cs.lane_creature.size() * sizeof(int), cs.stream));     // "unpublished" markers
        if (trace) {
            const size_t tb = (size_t)std::max(cs.n_members, 1) * 4 * sizeof(unsigned int);
            CK(ensure(cs.b_ttrace, tb));
            CK(cudaMemsetAsync(cs.b_ttrace.p, 0, tb, cs.stream));
            const size_t bytes = (size_t)h->plan.grid[k] * REM2D_TRACE_SAMPLES * 2 * sizeof(unsigned int);
            CK(ensure(cs.b_trace, bytes));
            CK(cudaMemsetAsync(cs.b_trace.p, 0, bytes, cs.stream));
        }
        ParkPolicy park = park_policy(k);
        if (trace) park.trace = (unsigned int*)cs.b_trace.p;
        if (h->plan.grid2[k] > 0) { CK(cudaEventRecord(cs.done2, cs.stream)); CK(cudaStreamWaitEvent(cs.stream2, cs.done2, 0)); }   // queue / park counters are reset
        g_classes(k).episode(h->plan.image, h->plan.gs[k], widest_group_shift(k, h->plan.gs[k]), h->plan.grid[k], cs.stream, cs.d_state, cs.d_lane_creature, cs.n_members, cs.d_queue, h->dpop,
                             h->d_ter, h->d_consts, max_ticks, h->d_fitness, h->d_ticks, h->d_alive, h->d_status, h->d_counters,
                             park, cs.d_park_state, cs.d_park_creature, cs.d_park_count, stats_dest(h), policy_of(h));
        // Nothing reads this copy, but it shapes the tail launches: without it the bench population gets twice the tail
        // launches and the second EA generation evaluates 40 % slower (3.1 s against 2.2 s; B200 at 1000 W).
        CK(cudaMemcpyAsync(cs.h_park_count, cs.d_park_count, sizeof(int), cudaMemcpyDeviceToHost, cs.stream));
        CK(cudaEventRecord(cs.t_end, cs.stream));
        h->launches++;
    }
    // overflow waves (after ALL first launches, so that their CTAs queue behind them): the creatures a class could not seat
    // in its first round, on the columns behind the first launch's
    for (int oi = 0; oi < N_CLASSES && !lp.warp_mode; ++oi) {
        const int k = lp.order[oi];
        ClassState& cs = h->cls[k];
        if (!cs.n_batches || h->plan.grid2[k] <= 0) continue;
        const int gs = h->plan.gs[k];
        const size_t first_block = ((size_t)h->plan.grid[k] * (32 >> gs) + 31) / 32;
        g_classes(k).episode(h->plan.image, gs, widest_group_shift(k, gs), h->plan.grid2[k], cs.stream2, cs.d_state + first_block * g_classes(k).words * 32, cs.d_lane_creature, cs.n_members,
                             cs.d_queue, h->dpop, h->d_ter, h->d_consts, max_ticks, h->d_fitness, h->d_ticks, h->d_alive, h->d_status,
                             h->d_counters, park_policy(k), cs.d_park_state, cs.d_park_creature, cs.d_park_count, stats_dest(h),
                             policy_of(h));
        h->launches++;
    }
    CK(cudaGetLastError());
    if (lp.park_ticks > 0) {
        // Tail: while the episode kernels run, poll their park counters and hand newly parked creatures to the
        // warp-per-creature tail mode right away (pool of streams), so the sequential ticks of the longest-lived
        // creatures overlap the bulk instead of extending the run; the last launch of a class happens when its episode
        // kernel has finished.
        bool running[N_CLASSES];
        int launched[N_CLASSES], waited[N_CLASSES] = {};
        int n_running = 0;
        size_t rr = 0;
        h->tail_used.assign(h->tail_pool.size(), 0);
        auto idle_stream = [&]() -> cudaStream_t {
            for (size_t i = 0; i < h->tail_pool.size(); ++i) {
                const size_t s = (rr + i) % h->tail_pool.size();
                if (!h->tail_used[s] || cudaStreamQuery(h->tail_pool[s]) == cudaSuccess) { rr = s + 1; h->tail_used[s] = 1; return h->tail_pool[s]; }
            }
            cudaStream_t st = nullptr;
            // highest priority: tail CTAs are placed before the queued overflow-wave CTAs of the episode launches
            if (h->tail_pool.size() < 4096 && cudaStreamCreateWithPriority(&st, cudaStreamNonBlocking, h->prio_high) == cudaSuccess) {
                h->tail_pool.push_back(st); h->tail_used.push_back(1);
                return st;
            }
            cudaGetLastError();
            const size_t s = rr++ % h->tail_pool.size();      // cannot grow: queue behind a busy stream
            h->tail_used[s] = 1;
            return h->tail_pool[s];
        };
        for (int k = 0; k < N_CLASSES; ++k) { running[k] = h->cls[k].n_batches > 0; launched[k] = 0; n_running += running[k] ? 1 : 0; }
        while (n_running > 0) {
            bool finished_now[N_CLASSES];
            for (int k = 0; k < N_CLASSES; ++k) {
                finished_now[k] = false;
                if (!running[k]) continue;
                cudaError_t q = cudaStreamQuery(h->cls[k].stream);       // BEFORE reading the counter: no slot can be missed
                if (q == cudaSuccess && h->plan.grid2[k] > 0) q = cudaStreamQuery(h->cls[k].stream2);
                if (q == cudaSuccess) finished_now[k] = true;
                else if (q != cudaErrorNotReady) { h->err = std::string("episode kernel: ") + cudaGetErrorString(q); return REM2D_E_CUDA; }
                CK(cudaMemcpyAsync(&h->h_poll[k], h->cls[k].d_park_count, sizeof(int), cudaMemcpyDeviceToHost, h->poll_stream));
            }
            CK(cudaStreamSynchronize(h->poll_stream));
            for (int k = N_CLASSES - 1; k >= 0; --k) {
                if (!running[k]) continue;
                ClassState& cs = h->cls[k];
                const int cnt = h->h_poll[k];
                // early launches in chunks (a handful of creatures or whatever is there when the class is done)
                if (cnt > launched[k]) ++waited[k]; else waited[k] = 0;
                if (cnt > launched[k] && (finished_now[k] || cnt - launched[k] >= 4 || waited[k] >= 3)) {
                    waited[k] = 0;
                    // a handful of parked creatures (random populations): a warp each; dozens at once (evolved populations,
                    // where many creatures outlive the threshold): 8 lanes each - 4x fewer warps at nearly the same tick latency
                    const int tail_gs = (cnt - launched[k] >= 32) ? std::min(3, h->opt.tail_group_shift) : h->opt.tail_group_shift;
                    g_classes(k).tail(h->plan.image, tail_gs, widest_group_shift(k, tail_gs), idle_stream(), cs.d_park_state, cs.d_park_creature, launched[k], cnt - launched[k],
                                      h->d_ter, h->d_consts, max_ticks, h->d_fitness, h->d_ticks, h->d_alive, h->d_status, h->d_counters,
                                      trace ? (unsigned int*)cs.b_ttrace.p : nullptr, stats_dest(h), policy_of(h));
                    CK(cudaGetLastError());
                    h->launches++;
                    launched[k] = cnt;
                }
                if (finished_now[k]) { running[k] = false; --n_running; }
            }
            if (n_running > 0) std::this_thread::sleep_for(std::chrono::microseconds(500));
        }
        for (size_t s = 0; s < h->tail_pool.size(); ++s) {
            if (!h->tail_used[s]) continue;
            CK(cudaEventRecord(h->pool_done, h->tail_pool[s]));
            CK(cudaStreamWaitEvent(h->user_stream, h->pool_done, 0));
        }
    }
    rc = join_streams(h);
    if (rc) return rc;
    rc = promote_overflowed(h, max_ticks);
    if (rc) return rc;
    CK(cudaEventRecord(h->ev_stop, h->user_stream));
    h->state_valid = false; h->results_valid = true; h->stats_valid = h->upload_stats;
    return REM2D_OK;
}

extern "C" int rem2d_reset(rem2d_handle* h) {
    if (!h) return REM2D_E_INVALID;
    if (!h->have_pop) { h->err = "reset: no population uploaded"; return REM2D_E_INVALID; }
    cudaSetDevice(h->cfg.device);
    return launch_reset(h);
}

static int gather(rem2d_handle* h) {
    if (!h->state_valid && !h->results_valid) { h->err = "no results: call rem2d_reset/rem2d_step or rem2d_run_episodes first"; return REM2D_E_INVALID; }
    for (int k = 0; k < N_CLASSES && h->state_valid; ++k) {
        ClassState& cs = h->cls[k];
        if (!cs.n_batches) continue;
        int n_lanes = cs.n_batches * 32;
        gather_kernel<<<(n_lanes + 127) / 128, 128, 0, h->user_stream>>>(cs.d_state, cs.d_lane_creature, n_lanes, g_classes(k).words,
                                                                        h->d_fitness, h->d_ticks, h->d_alive, h->d_status);
        h->launches++;
    }
    CK(cudaGetLastError());
    int n = h->n_creatures;
    CK(cudaMemcpyAsync(h->h_fitness.data(), h->d_fitness, sizeof(double) * n, cudaMemcpyDeviceToHost, h->user_stream));
    CK(cudaMemcpyAsync(h->h_ticks.data(), h->d_ticks, sizeof(int) * n, cudaMemcpyDeviceToHost, h->user_stream));
    CK(cudaMemcpyAsync(h->h_alive.data(), h->d_alive, sizeof(int) * n, cudaMemcpyDeviceToHost, h->user_stream));
    CK(cudaMemcpyAsync(h->h_status.data(), h->d_status, sizeof(int) * n, cudaMemcpyDeviceToHost, h->user_stream));
    CK(cudaStreamSynchronize(h->user_stream));
    for (int c = 0; c < n; ++c)
        if (h->h_status[c]) {
            char buf[200];
            snprintf(buf, sizeof(buf), "creature %d exceeded a capacity of its class (status %d: 1 contact pool, 4 TOI island)", c, h->h_status[c]);
            h->err = buf;
            return REM2D_E_CAPACITY;
        }
    return REM2D_OK;
}

// The stepping path: every class on its own stream, from the static creature -> column mapping. targets == nullptr: the sine
// controllers (step_kernel), or the policy of a population uploaded with one (step_kernel_policy, include/rem2d_policy.h);
// otherwise the host array of n_joints target angles (step_kernel_targets, include/rem2d_control.h), which overrides both.
static int launch_step(rem2d_handle* h, int32_t n_ticks, const double* targets) {
    if (!h->have_pop || n_ticks < 0) { h->err = "step: no population / negative tick count"; return REM2D_E_INVALID; }
    if (!h->state_valid) { h->err = "step: per-creature state was consumed by rem2d_run_episodes/rem2d_evaluate; call rem2d_reset first"; return REM2D_E_INVALID; }
    cudaSetDevice(h->cfg.device);
    h->stats_valid = false;                      // the stepping path records no statistics
    CK(cudaEventRecord(h->ev_start, h->user_stream));
    const double* d_targets = nullptr;
    if (targets) {
        CK(ensure(h->b_targets, sizeof(double) * (size_t)std::max(h->n_joints, 1)));
        d_targets = (const double*)h->b_targets.p;
        if (h->n_joints) CK(cudaMemcpyAsync(h->b_targets.p, targets, sizeof(double) * h->n_joints, cudaMemcpyHostToDevice, h->user_stream));
    }
    int rc = fork_streams(h);
    if (rc) return rc;
    for (int k = N_CLASSES - 1; k >= 0; --k) {        // most expensive class first
        ClassState& cs = h->cls[k];
        if (!cs.n_batches) continue;
        if (targets)
            g_classes(k).step_targets(step_group_shift(h->load, k, h->opt), cs.n_batches, cs.stream, cs.d_state, n_ticks, h->d_ter, h->d_consts,
                                      h->d_counters, cs.d_lane_creature, h->dpop.body_off, d_targets);
        else if (h->upload_policy)
            g_classes(k).step_policy(step_group_shift(h->load, k, h->opt), cs.n_batches, cs.stream, cs.d_state, n_ticks, h->d_ter, h->d_consts,
                                     h->d_counters, cs.d_lane_creature, h->dpolicy);
        else
            g_classes(k).step(step_group_shift(h->load, k, h->opt), cs.n_batches, cs.stream, cs.d_state, n_ticks, h->d_ter, h->d_consts, h->d_counters);
        h->launches++;
    }
    CK(cudaGetLastError());
    rc = join_streams(h);
    if (rc) return rc;
    CK(cudaEventRecord(h->ev_stop, h->user_stream));
    CK(cudaEventSynchronize(h->ev_stop));
    CK(cudaEventElapsedTime(&h->last_ms, h->ev_start, h->ev_stop));
    return REM2D_OK;
}

extern "C" {

int rem2d_step(rem2d_handle* h, int32_t n_ticks) {
    if (!h) return REM2D_E_INVALID;
    return launch_step(h, n_ticks, nullptr);
}

int rem2d_step_targets(rem2d_handle* h, const double* targets, int32_t n_ticks) {
    if (!h) return REM2D_E_INVALID;
    if (!targets) { h->err = "step_targets: NULL targets"; return REM2D_E_INVALID; }
    if (h->have_pop)
        for (int j = 0; j < h->n_joints; ++j)
            if (!std::isfinite(targets[j])) { h->err = "step_targets: target " + std::to_string(j) + " is not finite"; return REM2D_E_INVALID; }
    return launch_step(h, n_ticks, targets);
}

int rem2d_fitness(rem2d_handle* h, double* out) {
    if (!h || !out) return REM2D_E_INVALID;
    if (!h->have_pop) { h->err = "fitness: no population uploaded"; return REM2D_E_INVALID; }
    cudaSetDevice(h->cfg.device);
    int rc = gather(h);
    if (rc) return rc;
    memcpy(out, h->h_fitness.data(), sizeof(double) * h->n_creatures);
    return REM2D_OK;
}

int rem2d_get_counters(rem2d_handle* h, uint64_t* out) {
    if (!h || !out) return REM2D_E_INVALID;
    cudaSetDevice(h->cfg.device);
    CK(cudaStreamSynchronize(h->user_stream));
    CK(cudaMemcpy(out, h->d_counters, sizeof(unsigned long long) * REM2D_N_COUNTERS, cudaMemcpyDeviceToHost));
    return REM2D_OK;
}
// Diagnostics (libraries built with -DREM2D_PHASE_TIMING): warp-cycles per tick phase of the last evaluation,
// out[(mode * 6 + gs) * 16 + phase], mode 0 = queue launches, 1 = tail launches; zeros in production builds.
int rem2d_debug_phases(rem2d_handle* h, uint64_t* out) {
    if (!h || !out) return REM2D_E_INVALID;
    cudaSetDevice(h->cfg.device);
    CK(cudaStreamSynchronize(h->user_stream));
    CK(cudaMemcpy(out, h->d_counters + REM2D_N_COUNTERS, sizeof(unsigned long long) * 12 * 16, cudaMemcpyDeviceToHost));
    return REM2D_OK;
}

int rem2d_run_episodes(rem2d_handle* h, int32_t max_ticks) {
    if (!h) return REM2D_E_INVALID;
    if (!h->have_pop || max_ticks < 0) { h->err = "run_episodes: no population / negative tick count"; return REM2D_E_INVALID; }
    cudaSetDevice(h->cfg.device);
    int rc = launch_episodes(h, max_ticks);
    if (rc) return rc;
    CK(cudaEventSynchronize(h->ev_stop));
    CK(cudaEventElapsedTime(&h->last_ms, h->ev_start, h->ev_stop));
    return REM2D_OK;
}

int rem2d_ticks(rem2d_handle* h, int32_t* out) {
    if (!h || !out) return REM2D_E_INVALID;
    if (!h->have_pop) { h->err = "ticks: no population uploaded"; return REM2D_E_INVALID; }
    cudaSetDevice(h->cfg.device);
    int rc = gather(h);
    if (rc) return rc;
    memcpy(out, h->h_ticks.data(), sizeof(int) * h->n_creatures);
    return REM2D_OK;
}

int rem2d_evaluate(rem2d_handle* h, const rem2d_population* pop, int32_t max_ticks, double* fitness_out, int32_t* ticks_out) {
    int rc = upload_impl(h, pop, false);      // the episode kernel builds the worlds itself
    if (rc) return rc;
    rc = rem2d_run_episodes(h, max_ticks);
    if (rc) return rc;
    rc = gather(h);
    if (rc) return rc;
    if (fitness_out) memcpy(fitness_out, h->h_fitness.data(), sizeof(double) * h->n_creatures);
    if (ticks_out) memcpy(ticks_out, h->h_ticks.data(), sizeof(int) * h->n_creatures);
    return REM2D_OK;
}

// Measured non-fused FP32 issue peak of this device in GFLOP/s (best of 5), for the roofline denominator.
int rem2d_measure_fp32_peak(rem2d_handle* h, double* gflops) {
    if (!h || !gflops) return REM2D_E_INVALID;
    cudaSetDevice(h->cfg.device);
    int sms = 0;
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->cfg.device));
    const int blocks = sms * 8, threads = 256, iters = 1 << 14;
    float* d = nullptr;
    CK(cudaMalloc(&d, sizeof(float) * blocks * threads));
    double best = 0.0;
    for (int r = 0; r < 6; ++r) {
        CK(cudaEventRecord(h->ev_start, h->user_stream));
        fp32_issue_kernel<<<blocks, threads, 0, h->user_stream>>>(d, iters, 1.0000001f, 1e-7f);
        CK(cudaEventRecord(h->ev_stop, h->user_stream));
        CK(cudaEventSynchronize(h->ev_stop));
        float ms = 0.0f;
        CK(cudaEventElapsedTime(&ms, h->ev_start, h->ev_stop));
        double gf = (double)blocks * threads * iters * 16.0 / (ms * 1e-3) / 1e9;
        if (r > 0 && gf > best) best = gf;
    }
    cudaFree(d);
    *gflops = best;
    return REM2D_OK;
}

// Diagnostics: per capacity class, [nb, members, resident warps, kernel begin ms, kernel end ms] of the last
// rem2d_run_episodes (refill mode), times relative to its start. out has room for 5 * 16 floats; returns #classes.
int rem2d_debug_class_timeline(rem2d_handle* h, float* out) {
    if (!h || !out) return REM2D_E_INVALID;
    cudaSetDevice(h->cfg.device);
    cudaDeviceSynchronize();
    for (int k = 0; k < N_CLASSES; ++k) {
        ClassState& cs = h->cls[k];
        float b = -1.0f, e = -1.0f;
        if (cs.n_batches) { cudaEventElapsedTime(&b, h->ev_start, cs.t_begin); cudaEventElapsedTime(&e, h->ev_start, cs.t_end); }
        out[5 * k] = (float)class_dims[k].nb; out[5 * k + 1] = (float)cs.n_members; out[5 * k + 2] = (float)h->plan.grid[k];
        out[5 * k + 3] = b; out[5 * k + 4] = e;
    }
    cudaGetLastError();
    return N_CLASSES;
}

// Diagnostics: the REM2D_TRACE=1 samples of class k of the last rem2d_run_episodes: [warps][REM2D_TRACE_SAMPLES][2] uint32.
// Returns the number of warps (0: none), negative on error; copies at most max_words words.
int rem2d_debug_trace(rem2d_handle* h, int k, unsigned int* out, int64_t max_words) {
    if (!h || !out || k < 0 || k >= N_CLASSES) return REM2D_E_INVALID;
    ClassState& cs = h->cls[k];
    if (!cs.b_trace.p || !cs.n_batches) return 0;
    cudaSetDevice(h->cfg.device);
    cudaDeviceSynchronize();
    size_t words = (size_t)h->plan.grid[k] * REM2D_TRACE_SAMPLES * 2;
    if ((int64_t)words > max_words) words = (size_t)max_words;
    CK(cudaMemcpy(out, cs.b_trace.p, words * sizeof(unsigned int), cudaMemcpyDeviceToHost));
    return h->plan.grid[k];
}

// Diagnostics: per park slot {us parked, us tail start, us tail end, tail ticks} of class k (REM2D_TRACE=1). Returns #slots.
int rem2d_debug_tail_trace(rem2d_handle* h, int k, unsigned int* out, int64_t max_words) {
    if (!h || !out || k < 0 || k >= N_CLASSES) return REM2D_E_INVALID;
    ClassState& cs = h->cls[k];
    if (!cs.b_ttrace.p || !cs.n_batches) return 0;
    cudaSetDevice(h->cfg.device);
    cudaDeviceSynchronize();
    int parked = 0;
    CK(cudaMemcpy(&parked, cs.d_park_count, sizeof(int), cudaMemcpyDeviceToHost));
    size_t words = (size_t)parked * 4;
    if ((int64_t)words > max_words) words = (size_t)max_words;
    CK(cudaMemcpy(out, cs.b_ttrace.p, words * sizeof(unsigned int), cudaMemcpyDeviceToHost));
    return parked;
}

int rem2d_set_stats(rem2d_handle* h, int32_t on) {
    if (!h) return REM2D_E_INVALID;
    h->stats_on = on != 0;
    return REM2D_OK;
}

int rem2d_read_stats(rem2d_handle* h, rem2d_episode_stats* out) {
    if (!h || !out) return REM2D_E_INVALID;
    if (!h->stats_valid) {
        h->err = "read_stats: no statistics: run rem2d_run_episodes / rem2d_evaluate on a population uploaded with rem2d_set_stats(1)";
        return REM2D_E_INVALID;
    }
    cudaSetDevice(h->cfg.device);
    const size_t n = (size_t)h->n_creatures, nb = (size_t)h->n_bodies;
    const EpisodeStats& d = h->dstats;
    auto copy = [&](void* dst, const void* src, size_t bytes) {
        return dst && bytes ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, h->user_stream) : cudaSuccess;
    };
    CK(copy(out->end_reason, d.end_reason, n * sizeof(int32_t)));
    CK(copy(out->max_x, d.max_x, n * sizeof(float)));
    CK(copy(out->joint_work, d.joint_work, n * sizeof(double)));
    CK(copy(out->airborne_ticks, d.airborne_ticks, n * sizeof(int32_t)));
    CK(copy(out->ground_ticks, d.ground_ticks, nb * sizeof(int32_t)));
    CK(cudaStreamSynchronize(h->user_stream));
    return REM2D_OK;
}

int rem2d_set_policy(rem2d_handle* h, const double* weights, int32_t n_joints, int32_t n_hidden) {
    if (!h) return REM2D_E_INVALID;
    if (!weights) { h->policy_on = false; h->policy_w.clear(); h->policy_nj = h->policy_hidden = 0; return REM2D_OK; }
    if (n_hidden < 1 || n_hidden > REM2D_POLICY_MAX_HIDDEN || n_joints < 0) {
        h->err = "set_policy: need 1 <= n_hidden <= 16 and n_joints >= 0";
        return REM2D_E_INVALID;
    }
    const size_t n = (size_t)n_joints * (size_t)(10 * n_hidden + 1);
    for (size_t i = 0; i < n; ++i)
        if (!std::isfinite(weights[i])) { h->err = "set_policy: weight " + std::to_string(i) + " is not finite"; return REM2D_E_INVALID; }
    h->policy_w.assign(weights, weights + n);
    h->policy_nj = n_joints; h->policy_hidden = n_hidden; h->policy_on = true;
    return REM2D_OK;
}

int rem2d_set_priority(rem2d_handle* h, const float* expected_ticks, int32_t n) {
    if (!h || n < 0) return REM2D_E_INVALID;
    if (!expected_ticks || n == 0) h->priority.clear();
    else h->priority.assign(expected_ticks, expected_ticks + n);
    return REM2D_OK;
}

int rem2d_read_roots(rem2d_handle* h, float* root_x, double* wod, int32_t* alive) {
    if (!h) return REM2D_E_INVALID;
    if (!h->have_pop) { h->err = "read_roots: no population uploaded"; return REM2D_E_INVALID; }
    if (!h->state_valid) { h->err = "read_roots: per-creature state was consumed by rem2d_run_episodes; call rem2d_reset first"; return REM2D_E_INVALID; }
    cudaSetDevice(h->cfg.device);
    const size_t n = (size_t)std::max(h->n_creatures, 1);
    CK(ensure(h->b_roots, n * (sizeof(double) + sizeof(float) + sizeof(int))));
    double* d_wod = (double*)h->b_roots.p;
    float* d_x = (float*)(d_wod + n);
    int* d_alive = (int*)(d_x + n);
    for (int k = 0; k < N_CLASSES; ++k) {
        ClassState& cs = h->cls[k];
        if (!cs.n_batches) continue;
        const int n_lanes = cs.n_batches * 32;
        roots_kernel<<<(n_lanes + 127) / 128, 128, 0, h->user_stream>>>(cs.d_state, cs.d_lane_creature, n_lanes, g_classes(k).words, d_x, d_wod, d_alive);
        h->launches++;
    }
    CK(cudaGetLastError());
    if (root_x) CK(cudaMemcpyAsync(root_x, d_x, sizeof(float) * h->n_creatures, cudaMemcpyDeviceToHost, h->user_stream));
    if (wod) CK(cudaMemcpyAsync(wod, d_wod, sizeof(double) * h->n_creatures, cudaMemcpyDeviceToHost, h->user_stream));
    if (alive) CK(cudaMemcpyAsync(alive, d_alive, sizeof(int) * h->n_creatures, cudaMemcpyDeviceToHost, h->user_stream));
    CK(cudaStreamSynchronize(h->user_stream));
    return REM2D_OK;
}

int rem2d_read_observations(rem2d_handle* h, rem2d_observation* out) {
    if (!h || !out) return REM2D_E_INVALID;
    if (!h->have_pop) { h->err = "read_observations: no population uploaded"; return REM2D_E_INVALID; }
    if (!h->state_valid) { h->err = "read_observations: per-creature state was consumed by rem2d_run_episodes; call rem2d_reset first"; return REM2D_E_INVALID; }
    cudaSetDevice(h->cfg.device);
    const size_t n = (size_t)h->n_creatures, nb = (size_t)h->n_bodies, nj = (size_t)h->n_joints;
    CK(ensure(h->b_obs, sizeof(float) * (2 * nj + 6 * n) + sizeof(int32_t) * nb + 64));
    float* d_angle = (float*)h->b_obs.p;
    float* d_speed = d_angle + nj;
    float* d_root = d_speed + nj;
    int32_t* d_ground = (int32_t*)(d_root + 6 * n);
    for (int k = 0; k < N_CLASSES; ++k) {
        ClassState& cs = h->cls[k];
        if (!cs.n_batches) continue;
        const int n_lanes = cs.n_batches * 32;
        observations_kernel<<<(n_lanes + 127) / 128, 128, 0, h->user_stream>>>(cs.d_state, cs.d_lane_creature, n_lanes, g_classes(k).L,
                                                                               h->dpop.body_off, d_angle, d_speed, d_root, d_ground);
        h->launches++;
    }
    CK(cudaGetLastError());
    auto copy = [&](void* dst, const void* src, size_t bytes) {
        return dst && bytes ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, h->user_stream) : cudaSuccess;
    };
    CK(copy(out->joint_angle, d_angle, nj * sizeof(float)));
    CK(copy(out->joint_speed, d_speed, nj * sizeof(float)));
    CK(copy(out->root, d_root, 6 * n * sizeof(float)));
    CK(copy(out->ground, d_ground, nb * sizeof(int32_t)));
    CK(cudaStreamSynchronize(h->user_stream));
    return REM2D_OK;
}

float rem2d_last_step_ms(rem2d_handle* h) { return h ? h->last_ms : 0.0f; }
int64_t rem2d_launch_count(rem2d_handle* h) { return h ? h->launches : 0; }

// Test/diagnostic path: copies the whole state of every class to the host and decodes it there.
int rem2d_read_state(rem2d_handle* h, rem2d_state_view* out) {
    if (!h || !out) return REM2D_E_INVALID;
    if (!h->have_pop) { h->err = "read_state: no population uploaded"; return REM2D_E_INVALID; }
    if (!h->state_valid) { h->err = "read_state: per-creature state was consumed by rem2d_run_episodes; call rem2d_reset first"; return REM2D_E_INVALID; }
    cudaSetDevice(h->cfg.device);
    CK(cudaStreamSynchronize(h->user_stream));
    for (int k = 0; k < N_CLASSES; ++k) {
        ClassState& cs = h->cls[k];
        if (!cs.n_batches) continue;
        const ClassOps& ci = g_classes(k);
        std::vector<float> st((size_t)cs.n_batches * ci.words * 32);
        CK(cudaMemcpy(st.data(), cs.d_state, st.size() * sizeof(float), cudaMemcpyDeviceToHost));
        auto asint = [](float f) { int i; memcpy(&i, &f, 4); return i; };
        for (size_t gl = 0; gl < cs.lane_creature.size(); ++gl) {
            int c = cs.lane_creature[gl];
            if (c < 0) continue;
            const float* g = st.data() + (gl >> 5) * (size_t)ci.words * 32 + (gl & 31);
            auto S = [&](int f) { return g[f * 32]; };
            auto B = [&](int f, int i) { return g[(ci.off_body + i * BF_COUNT + f) * 32]; };
            auto J = [&](int f, int j) { return g[(ci.off_joint + j * JF_COUNT + f) * 32]; };
            auto C = [&](int f, int q) { return g[(ci.off_cont + q * CF_COUNT + f) * 32]; };
            int b0 = h->body_off[c], nb = h->body_off[c + 1] - b0, j0 = b0 - c;
            int awake = 0;
            for (int i = 0; i < nb; ++i) {
                if (out->pose) { out->pose[3 * (b0 + i)] = B(BF_CX, i); out->pose[3 * (b0 + i) + 1] = B(BF_CY, i); out->pose[3 * (b0 + i) + 2] = B(BF_A, i); }
                if (out->vel) { out->vel[3 * (b0 + i)] = B(BF_VX, i); out->vel[3 * (b0 + i) + 1] = B(BF_VY, i); out->vel[3 * (b0 + i) + 2] = B(BF_W, i); }
                awake |= asint(B(BF_FLAGS, i)) & BFL_AWAKE;
            }
            for (int j = 0; j < nb - 1; ++j) {
                if (out->joint_impulse) {
                    float* o = &out->joint_impulse[4 * (j0 + j)];
                    o[0] = J(JF_IMPX, j); o[1] = J(JF_IMPY, j); o[2] = J(JF_IMPZ, j); o[3] = J(JF_MIMP, j);
                }
                if (out->limit_state) out->limit_state[j0 + j] = asint(J(JF_LIMIT, j));
                if (out->motor_speed) out->motor_speed[j0 + j] = J(JF_MSPEED, j);
            }
            if (out->alive) out->alive[c] = asint(S(S_ALIVE));
            if (out->ticks) out->ticks[c] = asint(S(S_TICKS));
            if (out->awake) out->awake[c] = awake ? 1 : 0;
            if (out->wod) { int lo = asint(S(S_WOD_LO)), hi = asint(S(S_WOD_HI)); uint64_t u = ((uint64_t)(uint32_t)hi << 32) | (uint32_t)lo; double d; memcpy(&d, &u, 8); out->wod[c] = d; }
            int nc = asint(S(S_NC)), ntouch = 0;
            for (int q = 0; q < nc; ++q) ntouch += ((asint(C(CF_KEY, q)) >> 16) & CK_TOUCHING) ? 1 : 0;
            if (out->n_contacts) out->n_contacts[c] = nc;
            if (out->n_touching) out->n_touching[c] = ntouch;
            if (out->touching_pairs && out->max_pairs > 0) {
                int32_t* tp = &out->touching_pairs[(size_t)c * out->max_pairs * 2];
                float* ti = out->touching_impulse ? &out->touching_impulse[(size_t)c * out->max_pairs * 4] : nullptr;
                for (int q = 0; q < out->max_pairs * 2; ++q) tp[q] = -1;
                if (ti) for (int q = 0; q < out->max_pairs * 4; ++q) ti[q] = 0.0f;
                std::vector<std::pair<int, int>> pairs;    // (body<<8 | edge, pool index)
                for (int q = 0; q < nc; ++q) {
                    int key = asint(C(CF_KEY, q));
                    if (!((key >> 16) & CK_TOUCHING)) continue;
                    pairs.push_back({((key & 0xff) << 8) | ((key >> 8) & 0xff), q});
                }
                std::sort(pairs.begin(), pairs.end());
                for (size_t q = 0; q < pairs.size() && (int)q < out->max_pairs; ++q) {
                    int pq = pairs[q].second;
                    int key = asint(C(CF_KEY, pq));
                    int count = (key >> (16 + CK_COUNT_SHIFT)) & 3;
                    tp[2 * q] = key & 0xff; tp[2 * q + 1] = (key >> 8) & 0xff;
                    if (ti) {
                        ti[4 * q] = C(CF_P0N, pq); ti[4 * q + 1] = count > 1 ? C(CF_P1N, pq) : 0.0f;
                        ti[4 * q + 2] = C(CF_P0T, pq); ti[4 * q + 3] = count > 1 ? C(CF_P1T, pq) : 0.0f;
                    }
                }
            }
        }
    }
    return REM2D_OK;
}

}  // extern "C"
