// rem2d_probe.cu — TEST INFRASTRUCTURE: runs single geometry functions of gym_rem2d_b200/csrc/rem2d_device.cuh (the device
// code of the CUDA kernels) on batches of cases, so that tests/test_device_geometry.py can compare them with float64
// references. Each entry point calls the device code's own functions: rot_set, Sim::contact_update, Sim::gjk and
// Sim::time_of_impact. One case = one creature column with one body (body 0) and, for the narrow phase, one pool contact.
//
// The same source is built three times (Makefile): g++ -DREM2D_EMU -ffp-contract=off (the CPU build, through
// tests/emu/rem2d_emu_shim.h; one host thread runs the cases one after the other), nvcc -fmad=false (what the CUDA library
// runs) and nvcc -fmad=true (what Engine(precision="fast") runs). On the GPU every case is one thread with a group of one
// lane (gs = 0) and its own cold column; every call allocates, launches once, copies back and frees. Every entry point
// returns 0, or -1 on bad arguments, or a CUDA error code.
#include <cstdint>
#include <cstring>
#include <vector>

#ifdef REM2D_EMU
#include "../emu/rem2d_emu_shim.h"
#endif
#include "../../gym_rem2d_b200/csrc/rem2d_device.cuh"

#ifdef REM2D_EMU
thread_local emu::Ctx* emu::ctx = nullptr;
#endif

using namespace rem2d;

namespace {

struct BodyIn {            // per case: shape and pose of body 0 (a box of half extents hx, hy or a circle of radius hx)
    const int32_t* circle; const float *hx, *hy, *x, *y, *angle;
};
struct ContactIn {         // per case: edge index, old manifold (count, id0, id1) and old impulses (n0, t0, n1, t1)
    const int32_t* edge; const int32_t* old_i; const float* old_imp;
};
struct ContactOut {        // per case: count, type, touching, id0, id1 | ln.x, ln.y, lp.x, lp.y, p0, p1, n0, t0, n1, t1
    int32_t* out_i; float* out_f;
};
struct DistIn { const float* ev; const int32_t* cache_in; const float* metric_in; };      // ev: v1.x v1.y v2.x v2.y
struct DistOut { float* dist; int32_t* cache_out; float* metric_out; };                  // cache: count, ia[3], ib[3]
struct ToiIn { const float* ev; const float* sweep; };                                    // sweep: c0.x c0.y a0 c.x c.y a alpha0
struct ToiOut { int32_t* touching; float* t; };

const int NB = 1, NC = 1, NT = 1;

__device__ __forceinline__ void sim_init(Sim& sim, int i, float* cold, const Layout& L, const Terrain* ter, const Consts* k, float* hot) {
    sim.L = L;
    sim.set_group(0, i & 31, hot);
    sim.g = cold + (size_t)(i >> 5) * L.words * 32 + (i & 31);
    sim.ter = ter; sim.k = k;
    for (int c = 0; c < REM2D_N_COUNTERS; ++c) sim.cnt.c[c] = 0u;
    sim.nb = 1; sim.nj = 0;
}
// body 0 as build_world leaves it (at rest, awake), with its rotation cached by sync_transform
__device__ __forceinline__ void set_body(Sim& sim, const BodyIn& b, int i) {
    for (int f = 0; f < BF_COUNT; ++f) sim.B(f, 0) = 0.0f;
    sim.B(BF_CX, 0) = b.x[i]; sim.B(BF_CY, 0) = b.y[i]; sim.B(BF_A, 0) = b.angle[i];
    sim.B(BF_C0X, 0) = b.x[i]; sim.B(BF_C0Y, 0) = b.y[i]; sim.B(BF_A0, 0) = b.angle[i];
    sim.B(BF_HX, 0) = b.hx[i]; sim.B(BF_HY, 0) = b.hy[i];
    sim.setBi(BF_FLAGS, 0, BFL_AWAKE | (b.circle[i] ? BFL_CIRCLE : 0));
    sim.sync_transform(0);
}

__device__ __forceinline__ void case_rot_set(int i, const float* a, float* s, float* c) {
    Rot q = rot_set(a[i]);
    s[i] = q.s; c[i] = q.c;
}

__device__ __forceinline__ void case_contact(int i, float* cold, const Layout& L, const Terrain* ter, const Consts* k, float* hot,
                                             BodyIn b, ContactIn ci, ContactOut co) {
    Sim sim;
    sim_init(sim, i, cold, L, ter, k, hot);
    set_body(sim, b, i);
    for (int f = 0; f < CF_COUNT; ++f) sim.C(f, 0) = 0.0f;
    const int oc = ci.old_i[3 * i];
    int flags = CK_ENABLED | (oc > 0 ? CK_TOUCHING : 0) | (oc << CK_COUNT_SHIFT);
    sim.setCi(CF_KEY, 0, 0 | (ci.edge[i] << 8) | (flags << 16));
    sim.setCi(CF_P0ID, 0, ci.old_i[3 * i + 1]); sim.setCi(CF_P1ID, 0, ci.old_i[3 * i + 2]);
    sim.C(CF_P0N, 0) = ci.old_imp[4 * i]; sim.C(CF_P0T, 0) = ci.old_imp[4 * i + 1];
    sim.C(CF_P1N, 0) = ci.old_imp[4 * i + 2]; sim.C(CF_P1T, 0) = ci.old_imp[4 * i + 3];
    sim.setSi(S_NC, 1);
    sim.contact_update(0);
    const int key = sim.Ci(CF_KEY, 0), fl = (key >> 16) & 0xff;
    const int count = (fl >> CK_COUNT_SHIFT) & 3;
    int32_t* oi = co.out_i + 5 * i;
    float* of = co.out_f + 14 * i;
    oi[0] = count; oi[1] = (fl >> CK_TYPE_SHIFT) & 3; oi[2] = (fl & CK_TOUCHING) ? 1 : 0;
    oi[3] = sim.Ci(CF_P0ID, 0); oi[4] = sim.Ci(CF_P1ID, 0);
    const int fields[12] = { CF_LNX, CF_LNY, CF_LPX, CF_LPY, CF_P0X, CF_P0Y, CF_P1X, CF_P1Y, CF_P0N, CF_P0T, CF_P1N, CF_P1T };
    for (int f = 0; f < 12; ++f) of[f] = sim.C(fields[f], 0);
    of[12] = sim.B(BF_QS, 0); of[13] = sim.B(BF_QC, 0);
}

__device__ __forceinline__ void case_distance(int i, float* cold, const Layout& L, const Terrain* ter, const Consts* k, float* hot,
                                              BodyIn b, DistIn di, DistOut dout) {
    Sim sim;
    sim_init(sim, i, cold, L, ter, k, hot);
    set_body(sim, b, i);
    const float* e = di.ev + 4 * i;
    V2 ev[2] = { mk(e[0], e[1]), mk(e[2], e[3]) };
    Sim::Prox pb = sim.body_proxy(0);
    Rot q; q.s = sim.B(BF_QS, 0); q.c = sim.B(BF_QC, 0);
    V2 p = mk(sim.B(BF_CX, 0), sim.B(BF_CY, 0));
    Sim::SimplexCache cache;
    const int32_t* cin = di.cache_in + 7 * i;
    cache.count = cin[0]; cache.metric = di.metric_in[i];
    for (int j = 0; j < 3; ++j) { cache.ia[j] = cin[1 + j]; cache.ib[j] = cin[4 + j]; }
    dout.dist[i] = sim.gjk(cache, ev, pb, p, q);
    int32_t* cout = dout.cache_out + 7 * i;
    cout[0] = cache.count; dout.metric_out[i] = cache.metric;
    for (int j = 0; j < 3; ++j) { cout[1 + j] = j < cache.count ? cache.ia[j] : -1; cout[4 + j] = j < cache.count ? cache.ib[j] : -1; }
}

__device__ __forceinline__ void case_toi(int i, float* cold, const Layout& L, const Terrain* ter, const Consts* k, float* hot,
                                         BodyIn b, ToiIn ti, ToiOut to) {
    Sim sim;
    sim_init(sim, i, cold, L, ter, k, hot);
    set_body(sim, b, i);
    const float* e = ti.ev + 4 * i;
    const float* s = ti.sweep + 7 * i;
    V2 ev[2] = { mk(e[0], e[1]), mk(e[2], e[3]) };
    Sim::Prox pb = sim.body_proxy(0);                     // as contact_toi builds it
    Sim::Sweep sw;
    sw.c0 = mk(s[0], s[1]); sw.a0 = s[2]; sw.c = mk(s[3], s[4]); sw.a = s[5]; sw.alpha0 = s[6];
    float t;
    to.touching[i] = sim.time_of_impact(ev, pb, sw, t) ? 1 : 0;
    to.t[i] = t;
}

void fill_edges(Terrain* ter, const float* edges, int n_edges) {
    memset(ter, 0, sizeof(Terrain));
    ter->n_edges = n_edges;
    for (int j = 0; j < n_edges; ++j) {
        ter->v1x[j] = edges[4 * j]; ter->v1y[j] = edges[4 * j + 1]; ter->v2x[j] = edges[4 * j + 2]; ter->v2y[j] = edges[4 * j + 3];
    }
}

#ifdef REM2D_EMU
// ---------------------------------------------------------------- CPU: one host thread, cases in order
struct Run {
    Layout L = make_layout(NB, NC, NT);
    std::vector<float> cold;
    float hot[32] = {};
    Terrain ter;
    Consts k;
    emu::Warp warp;
    emu::Ctx ctx;
    explicit Run(int n) : cold((size_t)((n + 31) / 32) * make_layout(NB, NC, NT).words * 32, 0.0f) {
        memset(&ter, 0, sizeof(ter)); memset(&k, 0, sizeof(k));
        ctx.warp = &warp; ctx.lane = 0; memset(ctx.local_sense, 0, sizeof(ctx.local_sense));
        emu::ctx = &ctx;          // a group barrier reached by mistake is a one-lane barrier here, as on the GPU
    }
    ~Run() { emu::ctx = nullptr; }
};
#else
// ---------------------------------------------------------------- GPU: one thread per case, device 0
struct Dev {                      // device buffers of one call, freed by the destructor
    std::vector<void*> ptrs;
    cudaStream_t st = nullptr;
    cudaError_t err = cudaSuccess;
    Dev() { if (err == cudaSuccess) err = cudaSetDevice(0); if (err == cudaSuccess) err = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking); }
    ~Dev() { for (void* p : ptrs) cudaFree(p); if (st) cudaStreamDestroy(st); }
    template <class T> T* alloc(size_t n) {
        void* p = nullptr;
        if (err == cudaSuccess) err = cudaMalloc(&p, n * sizeof(T) > 0 ? n * sizeof(T) : 1);
        if (err == cudaSuccess) { ptrs.push_back(p); err = cudaMemsetAsync(p, 0, n * sizeof(T), st); }
        return (T*)p;
    }
    template <class T> const T* in(const T* h, size_t n) {
        T* d = alloc<T>(n);
        if (err == cudaSuccess) err = cudaMemcpyAsync(d, h, n * sizeof(T), cudaMemcpyHostToDevice, st);
        return d;
    }
    template <class T> void out(T* h, const T* d, size_t n) {
        if (err == cudaSuccess) err = cudaMemcpyAsync(h, d, n * sizeof(T), cudaMemcpyDeviceToHost, st);
    }
    int finish() {
        if (err == cudaSuccess) err = cudaStreamSynchronize(st);
        if (err == cudaSuccess) err = cudaGetLastError();
        return (int)err;
    }
    BodyIn body(const BodyIn& b, int n) {
        BodyIn d;
        d.circle = in(b.circle, n); d.hx = in(b.hx, n); d.hy = in(b.hy, n); d.x = in(b.x, n); d.y = in(b.y, n); d.angle = in(b.angle, n);
        return d;
    }
};

__global__ void k_rot_set(int n, const float* a, float* s, float* c) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) case_rot_set(i, a, s, c);
}
__global__ void k_contact(int n, float* cold, Layout L, const Terrain* ter, const Consts* k, BodyIn b, ContactIn ci, ContactOut co) {
    __shared__ float hot[32];
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) case_contact(i, cold, L, ter, k, hot, b, ci, co);
}
__global__ void k_distance(int n, float* cold, Layout L, const Terrain* ter, const Consts* k, BodyIn b, DistIn di, DistOut dout) {
    __shared__ float hot[32];
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) case_distance(i, cold, L, ter, k, hot, b, di, dout);
}
__global__ void k_toi(int n, float* cold, Layout L, const Terrain* ter, const Consts* k, BodyIn b, ToiIn ti, ToiOut to) {
    __shared__ float hot[32];
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) case_toi(i, cold, L, ter, k, hot, b, ti, to);
}
const int THREADS = 128;
inline int blocks(int n) { return (n + THREADS - 1) / THREADS; }
#endif

}  // namespace

extern "C" {

int probe_fmad() {
#if defined(REM2D_EMU)
    return 0;
#elif defined(REM2D_PROBE_FMAD)
    return 1;
#else
    return 0;
#endif
}

int probe_rot_set(int n, const float* a, float* s, float* c) {
    if (n < 1) return -1;
#ifdef REM2D_EMU
    Run r(1);
    for (int i = 0; i < n; ++i) case_rot_set(i, a, s, c);
    return 0;
#else
    Dev d;
    const float* da = d.in(a, n);
    float* ds = d.alloc<float>(n); float* dc = d.alloc<float>(n);
    if (d.err == cudaSuccess) { k_rot_set<<<blocks(n), THREADS, 0, d.st>>>(n, da, ds, dc); d.err = cudaGetLastError(); }
    d.out(s, ds, n); d.out(c, dc, n);
    return d.finish();
#endif
}

// edges: [n_edges][4] (v1.x, v1.y, v2.x, v2.y), the terrain table; edge[i] < n_edges picks the edge of case i.
// old_i: [n][3] old manifold count, id0, id1; old_imp: [n][4]. out_i: [n][5]; out_f: [n][14] (see ContactOut; the last two are
// the cached rotation q.s, q.c of the body).
int probe_contact_update(const float* edges, int n_edges, int n, const int32_t* edge, const int32_t* circle, const float* hx,
                         const float* hy, const float* x, const float* y, const float* angle, const int32_t* old_i,
                         const float* old_imp, int32_t* out_i, float* out_f) {
    if (n < 1 || n_edges < 1 || n_edges > RB_MAX_EDGES) return -1;
    for (int i = 0; i < n; ++i) if (edge[i] < 0 || edge[i] >= n_edges || old_i[3 * i] < 0 || old_i[3 * i] > 2) return -1;
    BodyIn b = { circle, hx, hy, x, y, angle };
#ifdef REM2D_EMU
    Run r(n);
    fill_edges(&r.ter, edges, n_edges);
    ContactIn ci = { edge, old_i, old_imp };
    ContactOut co = { out_i, out_f };
    for (int i = 0; i < n; ++i) case_contact(i, r.cold.data(), r.L, &r.ter, &r.k, r.hot, b, ci, co);
    return 0;
#else
    Terrain ter; fill_edges(&ter, edges, n_edges);
    Consts k; memset(&k, 0, sizeof(k));
    const Layout L = make_layout(NB, NC, NT);
    Dev d;
    float* cold = d.alloc<float>((size_t)blocks(n) * (THREADS / 32) * L.words * 32);
    const Terrain* dter = d.in(&ter, 1);
    const Consts* dk = d.in(&k, 1);
    BodyIn db = d.body(b, n);
    ContactIn ci = { d.in(edge, n), d.in(old_i, 3 * (size_t)n), d.in(old_imp, 4 * (size_t)n) };
    ContactOut co = { d.alloc<int32_t>(5 * (size_t)n), d.alloc<float>(14 * (size_t)n) };
    if (d.err == cudaSuccess) { k_contact<<<blocks(n), THREADS, 0, d.st>>>(n, cold, L, dter, dk, db, ci, co); d.err = cudaGetLastError(); }
    d.out(out_i, co.out_i, 5 * (size_t)n); d.out(out_f, co.out_f, 14 * (size_t)n);
    return d.finish();
#endif
}

// ev: [n][4] edge of each case; cache_in: [n][7] (count, ia[3], ib[3]; count 0 = cold start), metric_in: [n].
int probe_distance(int n, const float* ev, const int32_t* circle, const float* hx, const float* hy, const float* x, const float* y,
                   const float* angle, const int32_t* cache_in, const float* metric_in, float* dist, int32_t* cache_out,
                   float* metric_out) {
    if (n < 1) return -1;
    for (int i = 0; i < n; ++i) {
        const int32_t* c = cache_in + 7 * i;
        if (c[0] < 0 || c[0] > 3) return -1;
        for (int j = 0; j < c[0]; ++j) if (c[1 + j] < 0 || c[1 + j] > 1 || c[4 + j] < 0 || c[4 + j] > (circle[i] ? 0 : 3)) return -1;
    }
    BodyIn b = { circle, hx, hy, x, y, angle };
#ifdef REM2D_EMU
    Run r(n);
    DistIn di = { ev, cache_in, metric_in };
    DistOut dout = { dist, cache_out, metric_out };
    for (int i = 0; i < n; ++i) case_distance(i, r.cold.data(), r.L, &r.ter, &r.k, r.hot, b, di, dout);
    return 0;
#else
    const Layout L = make_layout(NB, NC, NT);
    Dev d;
    float* cold = d.alloc<float>((size_t)blocks(n) * (THREADS / 32) * L.words * 32);
    BodyIn db = d.body(b, n);
    DistIn di = { d.in(ev, 4 * (size_t)n), d.in(cache_in, 7 * (size_t)n), d.in(metric_in, n) };
    DistOut dout = { d.alloc<float>(n), d.alloc<int32_t>(7 * (size_t)n), d.alloc<float>(n) };
    if (d.err == cudaSuccess) { k_distance<<<blocks(n), THREADS, 0, d.st>>>(n, cold, L, nullptr, nullptr, db, di, dout); d.err = cudaGetLastError(); }
    d.out(dist, dout.dist, n); d.out(cache_out, dout.cache_out, 7 * (size_t)n); d.out(metric_out, dout.metric_out, n);
    return d.finish();
#endif
}

// ev: [n][4]; sweep: [n][7] (c0.x, c0.y, a0, c.x, c.y, a, alpha0) of body 0 (x, y, angle of BodyIn are unused by the query).
int probe_toi(int n, const float* ev, const int32_t* circle, const float* hx, const float* hy, const float* sweep, int32_t* touching,
              float* t) {
    if (n < 1) return -1;
    std::vector<float> x(n), y(n), a(n);
    for (int i = 0; i < n; ++i) { x[i] = sweep[7 * i]; y[i] = sweep[7 * i + 1]; a[i] = sweep[7 * i + 2]; }
    BodyIn b = { circle, hx, hy, x.data(), y.data(), a.data() };
#ifdef REM2D_EMU
    Run r(n);
    ToiIn ti = { ev, sweep };
    ToiOut to = { touching, t };
    for (int i = 0; i < n; ++i) case_toi(i, r.cold.data(), r.L, &r.ter, &r.k, r.hot, b, ti, to);
    return 0;
#else
    const Layout L = make_layout(NB, NC, NT);
    Dev d;
    float* cold = d.alloc<float>((size_t)blocks(n) * (THREADS / 32) * L.words * 32);
    BodyIn db = d.body(b, n);
    ToiIn ti = { d.in(ev, 4 * (size_t)n), d.in(sweep, 7 * (size_t)n) };
    ToiOut to = { d.alloc<int32_t>(n), d.alloc<float>(n) };
    if (d.err == cudaSuccess) { k_toi<<<blocks(n), THREADS, 0, d.st>>>(n, cold, L, nullptr, nullptr, db, ti, to); d.err = cudaGetLastError(); }
    d.out(touching, to.touching, n); d.out(t, to.t, n);
    return d.finish();
#endif
}

}  // extern "C"
