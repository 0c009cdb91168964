// mfx_host.cpp -- host side of libmafrix_cuda: the C ABI (include/mafrix_cuda.h), the host
// reproductions of PinholeCamera and Bvh.Build, scene flattening into the two HBM layouts and
// the wavefront driver that sequences the kernels of mfx_exact.cu / mfx_fast.cu.
//
// Compiled with -ffp-contract=off: the flattening arithmetic (edge vectors, areas, camera
// basis) must round exactly like the reference's f64 expressions.
#include "../../include/mafrix_cuda.h"
#include "mfx_internal.h"
#include "mfx_build.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <future>
#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <vector>

// ------------------------------------------------------------------ errors
static thread_local std::string g_err;
#define fail mfx_fail
#define env_long mfx_env_long

int mfx_fail(int code, const char *fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CUDA_TRY(x)                                                                              \
    do {                                                                                         \
        cudaError_t e_ = (x);                                                                    \
        if (e_ != cudaSuccess)                                                                   \
            return fail(e_ == cudaErrorMemoryAllocation ? MFX_ERR_OUT_OF_MEMORY : MFX_ERR_CUDA,  \
                        "%s failed: %s (%s:%d)", #x, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

#define MFX_TRY(x)               \
    do {                         \
        int r_ = (x);            \
        if (r_ != MFX_OK) return r_; \
    } while (0)

#ifdef MFX_DEBUG_CHECKS
extern "C" const char *mfx_version(void) { return "mafrix_cuda 0.2 (sm_100a, DEBUG CHECKS)"; }
#else
extern "C" const char *mfx_version(void) { return "mafrix_cuda 0.2 (sm_100a)"; }
#endif
extern "C" const char *mfx_last_error(void) { return g_err.c_str(); }

extern "C" int mfx_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

static thread_local int g_device = -1;

extern "C" int mfx_init(int device)
{
    int n = mfx_device_count();
    if (n <= 0) return fail(MFX_ERR_NO_DEVICE, "no CUDA device visible: libmafrix_cuda has no CPU fallback");
    if (device < 0 || device >= n) return fail(MFX_ERR_INVALID_ARGUMENT, "device %d out of range (0..%d)", device, n - 1);
    CUDA_TRY(cudaSetDevice(device));
    g_device = device;
    return MFX_OK;
}

// mfx_scene_create runs on the device the calling thread chose with mfx_init (default 0) ...
static int ensure_device()
{
    if (g_device >= 0) { CUDA_TRY(cudaSetDevice(g_device)); return MFX_OK; }
    return mfx_init(0);
}
// ... every other entry point takes a handle and runs on the device THAT HANDLE lives on, whichever thread calls
// (a .NET thread-pool or render-callback thread never called mfx_init: its thread-local default must not win).
static int bind_device(int device)
{
    CUDA_TRY(cudaSetDevice(device));
    return MFX_OK;
}

// ------------------------------------------------------------------ host math (f64, reference order)
struct H3 { double x, y, z; };
static inline H3 h3(double x, double y, double z) { return H3{ x, y, z }; }
static inline H3 hsub(H3 a, H3 b) { return h3(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline H3 hadd(H3 a, H3 b) { return h3(a.x + b.x, a.y + b.y, a.z + b.z); }
static inline H3 hmul(H3 a, double s) { return h3(a.x * s, a.y * s, a.z * s); }
static inline H3 hcross(H3 a, H3 b) { return h3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
static inline double hlen(H3 a) { return std::sqrt(a.x * a.x + a.y * a.y + a.z * a.z); }
static inline H3 hnorm(H3 a)
{
    double l = hlen(a);
    if (l == 0.0) return h3(0, 0, 0);
    return h3(a.x / l, a.y / l, a.z / l);
}
static inline H3 hld(const double *p) { return h3(p[0], p[1], p[2]); }
static inline void hst(double *p, H3 v) { p[0] = v.x; p[1] = v.y; p[2] = v.z; }

// PinholeCamera(pos, dir, fov, aspect): Camera.fs:96-133
extern "C" int mfx_camera_pinhole(const double pos[3], const double dir[3], double fov, double aspect, MfxCamera *out)
{
    if (!pos || !dir || !out) return fail(MFX_ERR_INVALID_ARGUMENT, "mfx_camera_pinhole: null argument");
    const double PI = 3.14159265358979323846;
    H3 fwd = hnorm(hld(dir));                                   // CameraCoordinate(dir), Camera.fs:96-104
    H3 up0 = hnorm(h3(0, 1, 0));
    H3 hori = hcross(fwd, hnorm(up0));                          // not re-normalised (quirk Q5)
    H3 vert = hcross(hori, fwd);
    double hs = std::tan(0.5 * fov * PI / 360.);                // Camera.fs:125: effective FOV = fov/2
    double vs = hs / aspect;
    H3 up = hmul(vert, vs), right = hmul(hori, hs);
    H3 down = h3(-up.x, -up.y, -up.z);
    H3 p = hld(pos);
    // TopLeft(pos, 0.5) = pos + dist*forward - 0.5*right + 0.5*up, Camera.fs:110-111
    H3 tl = hadd(hsub(hadd(p, hmul(fwd, 0.5)), hmul(right, 0.5)), hmul(up, 0.5));
    hst(out->pos, p); hst(out->topleft, tl); hst(out->right, right); hst(out->down, down);
    return MFX_OK;
}

// RayTraceCamera(lookfrom, lookat, vup, vfov, aspect, aperture, focus_dist, t0, t1): RenderTest/Sample/RayTracing.fs:335-358
extern "C" int mfx_camera_lens(const double lookfrom[3], const double lookat[3], const double vup[3], double vfov,
                               double aspect, double aperture, double focus_dist, MfxLensCamera *out)
{
    if (!lookfrom || !lookat || !vup || !out) return fail(MFX_ERR_INVALID_ARGUMENT, "mfx_camera_lens: null argument");
    const double PI = 3.14159265358979323846;
    out->lens_radius = aperture / 2.0;                                   // :347
    const double theta = vfov * PI / 180.;
    const double half_height = std::tan(theta / 2.);
    const double half_width = aspect * half_height;
    const H3 origin = hld(lookfrom);
    const H3 w = hnorm(hsub(hld(lookfrom), hld(lookat)));                // :352-354
    const H3 u = hnorm(hcross(hld(vup), w));
    const H3 v = hnorm(hcross(w, u));
    // origin - focus_dist*half_width*u - focus_dist*half_height*v - focus_dist*w, :355
    const H3 p = hsub(hsub(hsub(origin, hmul(u, focus_dist * half_width)), hmul(v, focus_dist * half_height)), hmul(w, focus_dist));
    hst(out->origin, origin); hst(out->lower_left, p);
    hst(out->horizontal, hmul(u, 2. * focus_dist * half_width));         // :357-358
    hst(out->vertical, hmul(v, 2. * focus_dist * half_height));
    hst(out->u, u); hst(out->v, v);
    return MFX_OK;
}

// ------------------------------------------------------------------ scene
// One Sample call in flight: what launch_sample enqueued and finish_sample needs to turn into MfxStats.  Two slots, so
// the download of frame k (copy stream) runs beside the kernels of frame k+1 (mfx_pixel_integrator_sample_async).
struct Span { size_t a, b; int cls; };
struct FrameJob {
    bool active = false;
    int device = 0;
    std::vector<cudaEvent_t> events;         // timing + dependency events of this job (grown on demand, reused)
    std::vector<Span> spans;
    size_t e_begin = 0, e_end = 1;
    uint32_t launches = 0, l_ext = 0, l_sh = 0;
    unsigned long long *d_totals = nullptr;  // [8] rays / paths / watchdog / hybrid fixups
    TravCounters *d_ctr = nullptr;
    unsigned long long *h_totals = nullptr;  // pinned host mirrors, filled by async copies behind the kernels
    TravCounters *h_ctr = nullptr;
    cudaEvent_t done = nullptr;              // kernels + stat copies of the job finished (main stream)
    cudaEvent_t copied = nullptr;            // async only: the texture download finished (copy stream)
    bool has_copy = false;
};

struct OwnTreeHost;
struct MfxScene {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;          // shadow queries of bounce b run beside the closest hits of bounce b+1 (run_sample)
    float4 *sh2[3] = { nullptr, nullptr, nullptr };   // second shadow queue (sh_o, sh_d, sh_c) of the two-stream mode
    int sh2_P = 0;
    uint2 *spill2 = nullptr;                 // the shadow launches' own stack spill columns in that mode (sized like sf.stack_spill)
    std::vector<MfxPrim> prims;
    std::vector<MfxMaterial> mats;
    std::vector<MfxBvhNode> nodes;
    std::vector<int32_t> indices;
    MfxAreaLight light;
    MfxCamera camera;
    MfxLensCamera lens;                      // MFX_SKY_TRACER
    std::vector<double> perlin_rf;           // MFX_SKY_TRACER: 256 or empty
    std::vector<int32_t> perlin_perm;        //                 768 or empty
    int width = 0, height = 0, max_depth = 0, integrator = 0;
    bool in_process_replica = false;         // one of mfx_multi_create's replicas: the workers share one process and one tree cache
    int host_share = 1;                      // ranks known to share this host (MfxSampleParams.world): the tree builder
                                             // forks over hardware threads / host_share

    std::vector<std::pair<void *, size_t>> allocs;   // every device buffer of this scene
    bool x_ready = false, f_ready = false, fr_ready = false, wx_ready = false, wf_ready = false;
    SceneX sx; SceneF sf; SceneF sf_ref; WaveX wx; WaveF wf;     // sf: own SAH tree; sf_ref: reference-tree layout
    uint64_t x_bytes = 0, f_bytes = 0, fr_bytes = 0, h_bytes = 0;
    bool h_ready = false, wh_ready = false;  // hybrid (id-exact closest hit on the own tree): tables, f64 ray queue
    SceneH sh; WaveH wh; int wh_P = 0;
    std::shared_ptr<OwnTreeHost> own_host;   // the cached host half of the own tree this scene was flattened from
    std::vector<int> f_slot_prim;            // own-tree fast slot -> caller's primitive index, bit 30 = second half of a Rect
    MatF *d_matf = nullptr;
    float *d_perlin_rf = nullptr; int *d_perlin_perm = nullptr;
    double *d_pixsum = nullptr;          // [w*h][4] row-major sums
    double *d_color_wh = nullptr;        // Color[w,h]
    float4 *d_rgba = nullptr;            // row-major float4 (internal, when the caller gives none)
    FrameJob jobs[2];
    int job_head = 0, job_count = 0;         // outstanding async frames: jobs[job_head], jobs[(job_head + 1) % 2]
    cudaStream_t copy_stream = nullptr;      // texture downloads of async frames
    double *d_color_async[2] = { nullptr, nullptr };   // Color[w,h] per async slot
    std::map<std::tuple<int, int, int>, std::pair<int *, int>> tilemaps;
    MfxStats stats;
};

// Process-wide cache of large device buffers (per device, keyed by size): a host that rebuilds its
// Scene every frame (the e2e path of bench.py) must not pay cudaMalloc/cudaFree for ~0.5 GB of
// path state each time.  Bounded; everything beyond the bound is really freed.
#include <mutex>
#include <thread>
static std::mutex g_pool_mu;
static std::multimap<std::pair<int, size_t>, void *> g_pool;
static std::map<int, size_t> g_pool_bytes;                   // parked bytes PER DEVICE (a budget shared by eight devices with two frames in flight each overflowed)
static const size_t POOL_MIN = 0, POOL_ENTRIES = 4096;       // every buffer is pooled: a host that re-creates its Scene per frame pays no cudaMalloc / cudaFree
static size_t pool_max()      // per device: a third of it (B200: 60 GB -- holds one full 128 Mi-path wave with its hybrid buffers), at most 64 GB
{
    static size_t v = 0;
    if (!v) { size_t fr = 0, tot = 0; v = (cudaMemGetInfo(&fr, &tot) == cudaSuccess && tot) ? std::min(tot / 3, (size_t)64 << 30) : ((size_t)32 << 30); }
    return v;
}

static void pool_trim(int device);
static int dev_alloc(MfxScene *s, void **p, size_t bytes)
{
    bytes = bytes ? bytes : 16;
    if (bytes >= POOL_MIN) {
        std::lock_guard<std::mutex> g(g_pool_mu);
        auto it = g_pool.find({ s->device, bytes });
        if (it != g_pool.end()) {
            *p = it->second; g_pool.erase(it); g_pool_bytes[s->device] -= bytes;
            s->allocs.push_back({ *p, bytes });
            return MFX_OK;
        }
    }
    cudaError_t e = cudaMalloc(p, bytes);
    if (e == cudaErrorMemoryAllocation) {       // memory parked in the pool is not "in use": give it back and retry once
        cudaGetLastError();
        pool_trim(s->device);
        e = cudaMalloc(p, bytes);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(e == cudaErrorMemoryAllocation ? MFX_ERR_OUT_OF_MEMORY : MFX_ERR_CUDA, "cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
    }
    s->allocs.push_back({ *p, bytes });
    return MFX_OK;
}

static void dev_release(int device, void *p, size_t bytes)
{
    if (bytes >= POOL_MIN) {
        std::lock_guard<std::mutex> g(g_pool_mu);
        if (g_pool_bytes[device] + bytes <= pool_max() && g_pool.size() < POOL_ENTRIES) { g_pool.insert({ { device, bytes }, p }); g_pool_bytes[device] += bytes; return; }
    }
    cudaFree(p);
}

// frees every cached buffer of one device (called when an allocation fails before giving up on its size)
static void pool_trim(int device)
{
    std::lock_guard<std::mutex> g(g_pool_mu);
    for (auto it = g_pool.begin(); it != g_pool.end();) {
        if (it->first.first == device) { cudaFree(it->second); g_pool_bytes[device] -= it->first.second; it = g_pool.erase(it); }
        else ++it;
    }
}

// gives one buffer of the scene back (to the pool) before the scene dies: the wave state grows on demand
static void dev_free_one(MfxScene *s, void *p, bool to_pool = true)
{
    if (!p) return;
    for (size_t i = 0; i < s->allocs.size(); i++)
        if (s->allocs[i].first == p) {
            if (to_pool) dev_release(s->device, p, s->allocs[i].second); else cudaFree(p);
            s->allocs.erase(s->allocs.begin() + (long)i);
            return;
        }
}

// one pinned staging buffer per process for downloads into pageable caller memory
static void *g_pinned = nullptr;
static size_t g_pinned_bytes = 0;
template <typename T> static int dev_alloc_t(MfxScene *s, T **p, size_t count) { return dev_alloc(s, (void **)p, count * sizeof(T)); }

template <typename T> static int upload(MfxScene *s, T **dp, const std::vector<T> &h)
{
    MFX_TRY(dev_alloc_t(s, dp, h.size()));
    // pageable source: cudaMemcpyAsync returns once the data is staged, so `h` may die right after; the kernels that
    // read *dp run on the same stream -- no synchronisation needed here
    if (!h.empty()) CUDA_TRY(cudaMemcpyAsync(*dp, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, s->stream));
    return MFX_OK;
}

long mfx_env_long(const char *name, long dflt)
{
    const char *v = getenv(name);
    if (!v || !*v) return dflt;
    return atol(v);
}

static int stream_get(int device, cudaStream_t *out);

// A caller-supplied Bvh (nodes + indices) is indexed by the flatteners and by the kernels: reject anything that is not
// a permutation / a well-formed heap-indexed tree instead of reading out of bounds.
static int validate_tree(const std::vector<MfxBvhNode> &nodes, const std::vector<int32_t> &indices)
{
    const int n = (int)indices.size();
    std::vector<char> seen((size_t)n, 0);
    for (int i = 0; i < n; i++) {
        const int v = indices[i];
        if (v < 0 || v >= n || seen[v]) return fail(MFX_ERR_INVALID_ARGUMENT, "supplied tree: indices[%d] = %d is not part of a permutation of 0..%d", i, v, n - 1);
        seen[v] = 1;
    }
    std::vector<int> todo{ 0 };
    long covered = 0;
    while (!todo.empty()) {
        const int i = todo.back(); todo.pop_back();
        const MfxBvhNode &nd = nodes[i];
        if (nd.count <= 0 || nd.first < 0 || (long)nd.first + nd.count > n)
            return fail(MFX_ERR_INVALID_ARGUMENT, "supplied tree: node %d covers [%d, %d + %d) outside 0..%d", i, nd.first, nd.first, nd.count, n);
        if (nd.count <= MFX_LEAF_NODE_COUNT) { covered += nd.count; continue; }
        if ((size_t)(2 * (long)i + 2) >= nodes.size()) return fail(MFX_ERR_INVALID_ARGUMENT, "supplied tree: interior node %d has no child slots", i);
        todo.push_back(2 * i + 1); todo.push_back(2 * i + 2);
    }
    if (covered != n) return fail(MFX_ERR_INVALID_ARGUMENT, "supplied tree: its leaves cover %ld of %d primitives", covered, n);
    return MFX_OK;
}

extern "C" int mfx_scene_create(const MfxSceneDesc *d, MfxScene **out)
{
    if (!d || !out) return fail(MFX_ERR_INVALID_ARGUMENT, "mfx_scene_create: null argument");
    *out = nullptr;
    if (!d->prims || d->n_prims <= 0) return fail(MFX_ERR_INVALID_ARGUMENT, "scene has no primitives");
    if (d->n_prims >= (1 << 27)) return fail(MFX_ERR_UNSUPPORTED, "more than 2^27 primitives");
    if (!d->materials || d->n_materials <= 0) return fail(MFX_ERR_INVALID_ARGUMENT, "scene has no materials");
    if (d->width <= 0 || d->height <= 0) return fail(MFX_ERR_INVALID_ARGUMENT, "bad film size %dx%d", d->width, d->height);
    if (d->max_depth < 0 || d->max_depth >= MFX_MAX_VERTS) return fail(MFX_ERR_UNSUPPORTED, "max_depth %d outside 0..%d", d->max_depth, MFX_MAX_VERTS - 1);
    if (d->integrator != MFX_PATH_INTEGRATOR && d->integrator != MFX_NEW_PATH_TRACER && d->integrator != MFX_SKY_TRACER)
        return fail(MFX_ERR_INVALID_ARGUMENT, "unknown integrator %d", d->integrator);
    const bool sky = (d->integrator == MFX_SKY_TRACER);
    if (sky && !d->sky) return fail(MFX_ERR_INVALID_ARGUMENT, "MFX_SKY_TRACER needs MfxSceneDesc.sky (lens camera)");
    for (int i = 0; i < d->n_materials; i++) {
        const int k = d->materials[i].kind;
        if (k < 0 || k > MFX_LAMBERT_NOISE) return fail(MFX_ERR_INVALID_ARGUMENT, "material %d: unknown kind %d", i, k);
        if (sky && k == MFX_SPECTRANS) return fail(MFX_ERR_INVALID_ARGUMENT, "material %d: SpecularTransmission does not exist in the sphere sample (use MFX_DIELECTRIC)", i);
        if (!sky && k > MFX_SPECTRANS) return fail(MFX_ERR_INVALID_ARGUMENT, "material %d: kind %d only exists under MFX_SKY_TRACER", i, k);
        if (k == MFX_LAMBERT_NOISE && (!d->sky->perlin_ranfloat || !d->sky->perlin_perm))
            return fail(MFX_ERR_INVALID_ARGUMENT, "material %d: MFX_LAMBERT_NOISE needs the Perlin tables", i);
    }
    if (sky && d->sky->perlin_perm)
        for (int i = 0; i < 768; i++)
            if (d->sky->perlin_perm[i] < 0 || d->sky->perlin_perm[i] > 255) return fail(MFX_ERR_INVALID_ARGUMENT, "perlin_perm[%d] = %d outside 0..255", i, d->sky->perlin_perm[i]);
    for (int i = 0; i < d->n_prims; i++) {
        // the sphere sample's IHitAble list holds spheres only (RayTracing.fs:176-253; MovingSphere is not carried over)
        if (sky && (d->prims[i].kind != MFX_SPHERE || !(d->prims[i].v[3] > 0.)))
            return fail(MFX_ERR_UNSUPPORTED, "primitive %d: MFX_SKY_TRACER takes spheres with a positive radius only", i);
        if (d->prims[i].kind < 0 || d->prims[i].kind > 2) return fail(MFX_ERR_INVALID_ARGUMENT, "primitive %d: unknown kind %d", i, d->prims[i].kind);
        if (d->prims[i].material < 0 || d->prims[i].material >= d->n_materials)
            return fail(MFX_ERR_INVALID_ARGUMENT, "primitive %d: material %d outside the table of %d", i, d->prims[i].material, d->n_materials);
    }
    const int n_slots_in = 2 * d->n_prims - 1;
    if (d->nodes) {     // argument errors come before the device check (and need no GPU to be reported)
        if (d->n_node_slots != n_slots_in || !d->indices)
            return fail(MFX_ERR_INVALID_ARGUMENT, "supplied tree needs 2n-1 = %d node slots and an index array", n_slots_in);
        MFX_TRY(validate_tree(std::vector<MfxBvhNode>(d->nodes, d->nodes + n_slots_in), std::vector<int32_t>(d->indices, d->indices + d->n_prims)));
    }
    MFX_TRY(ensure_device());
    MfxScene *s = new MfxScene();
    s->device = g_device;
    {   // cudaGetDeviceProperties costs tens of ms per call: one attribute query, cached per device
        static std::map<int, int> sm_cache;
        std::lock_guard<std::mutex> g(g_pool_mu);
        auto it = sm_cache.find(s->device);
        if (it == sm_cache.end()) {
            int sms = 148;
            if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s->device) != cudaSuccess) { cudaGetLastError(); sms = 148; }
            it = sm_cache.emplace(s->device, sms).first;
        }
        s->sm_count = it->second;
    }
    s->prims.assign(d->prims, d->prims + d->n_prims);
    s->mats.assign(d->materials, d->materials + d->n_materials);
    s->light = d->light; s->camera = d->camera;
    memset(&s->lens, 0, sizeof(s->lens));
    if (sky) {
        s->lens = d->sky->camera;
        // the lens camera rides in the pinhole slots (see LensX): the seams and the kernels share one ray formula
        memcpy(s->camera.pos, s->lens.origin, 24); memcpy(s->camera.topleft, s->lens.lower_left, 24);
        memcpy(s->camera.right, s->lens.horizontal, 24); memcpy(s->camera.down, s->lens.vertical, 24);
        memset(&s->light, 0, sizeof(s->light));
        if (d->sky->perlin_ranfloat) s->perlin_rf.assign(d->sky->perlin_ranfloat, d->sky->perlin_ranfloat + 256);
        if (d->sky->perlin_perm) s->perlin_perm.assign(d->sky->perlin_perm, d->sky->perlin_perm + 768);
    }
    s->width = d->width; s->height = d->height; s->max_depth = d->max_depth; s->integrator = d->integrator;
    const int n_slots = 2 * d->n_prims - 1;
    s->nodes.resize(n_slots); s->indices.resize(d->n_prims);
    int rc = MFX_OK;
    if (d->nodes) {
        if (d->n_node_slots != n_slots || !d->indices) { delete s; return fail(MFX_ERR_INVALID_ARGUMENT, "supplied tree needs 2n-1 = %d node slots and an index array", n_slots); }
        memcpy(s->nodes.data(), d->nodes, sizeof(MfxBvhNode) * (size_t)n_slots);
        memcpy(s->indices.data(), d->indices, sizeof(int32_t) * (size_t)d->n_prims);
    } else rc = mfx_bvh_build(s->prims.data(), d->n_prims, s->nodes.data(), n_slots, s->indices.data());
    if (rc != MFX_OK) { delete s; return rc; }
    if (stream_get(s->device, &s->stream) != MFX_OK) { delete s; return fail(MFX_ERR_CUDA, "cudaStreamCreate failed"); }
    memset(&s->stats, 0, sizeof(s->stats));
    *out = s;
    return MFX_OK;
}

static void stat_block_put(void *p);

// Streams and events are recycled per device for the life of the process, like the device buffers: a host that re-creates
// its Scene every frame (and the eight replicas of a multi-GPU handle) would otherwise issue ~150 driver calls per scene
// for them, contending for the driver with the worker threads that are launching the previous frame's kernels.
static std::map<int, std::vector<cudaStream_t>> g_streams;
static std::map<std::pair<int, int>, std::vector<cudaEvent_t>> g_events;      // (device, timing?) -> free events
static int stream_get(int device, cudaStream_t *out)
{
    {
        std::lock_guard<std::mutex> g(g_pool_mu);
        auto &v = g_streams[device];
        if (!v.empty()) { *out = v.back(); v.pop_back(); return MFX_OK; }
    }
    CUDA_TRY(cudaStreamCreateWithFlags(out, cudaStreamNonBlocking));
    return MFX_OK;
}
static void stream_put(int device, cudaStream_t st)       // the caller has synchronised it
{
    if (!st) return;
    std::lock_guard<std::mutex> g(g_pool_mu);
    g_streams[device].push_back(st);
}
static int event_get(int device, bool timing, cudaEvent_t *out)
{
    {
        std::lock_guard<std::mutex> g(g_pool_mu);
        auto &v = g_events[{ device, timing ? 1 : 0 }];
        if (!v.empty()) { *out = v.back(); v.pop_back(); return MFX_OK; }
    }
    CUDA_TRY(cudaEventCreateWithFlags(out, timing ? cudaEventDefault : cudaEventDisableTiming));
    return MFX_OK;
}
static void event_put(int device, bool timing, cudaEvent_t e)
{
    if (!e) return;
    std::lock_guard<std::mutex> g(g_pool_mu);
    g_events[{ device, timing ? 1 : 0 }].push_back(e);
}

extern "C" int mfx_scene_destroy(MfxScene *s)
{
    if (!s) return MFX_OK;
    cudaSetDevice(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    if (s->copy_stream) { cudaStreamSynchronize(s->copy_stream); stream_put(s->device, s->copy_stream); }
    for (auto &a : s->allocs) dev_release(s->device, a.first, a.second);
    for (FrameJob &j : s->jobs) {
        for (cudaEvent_t e : j.events) event_put(s->device, true, e);
        event_put(s->device, false, j.done);
        event_put(s->device, false, j.copied);
        stat_block_put(j.h_totals);
    }
    if (s->stream2) { cudaStreamSynchronize(s->stream2); stream_put(s->device, s->stream2); }
    if (s->stream) stream_put(s->device, s->stream);
    delete s;
    return MFX_OK;
}

extern "C" int mfx_scene_get_bvh(const MfxScene *s, MfxBvhNode *nodes_out, int32_t *indices_out)
{
    if (!s || !nodes_out || !indices_out) return fail(MFX_ERR_INVALID_ARGUMENT, "mfx_scene_get_bvh: null argument");
    memcpy(nodes_out, s->nodes.data(), sizeof(MfxBvhNode) * s->nodes.size());
    memcpy(indices_out, s->indices.data(), sizeof(int32_t) * s->indices.size());
    return MFX_OK;
}

// ---- flatten: exact layout
static void tri_sample_x(TriSampleX &t, H3 v0, H3 v1, H3 v2)
{
    hst(t.v0, v0); hst(t.e1, hsub(v1, v0)); hst(t.e2, hsub(v2, v0));
}
static double tri_area(H3 v0, H3 v1, H3 v2)      // Trangle.fs:108-116: |e1 x e2| * 0.5
{
    return hlen(hcross(hsub(v1, v0), hsub(v2, v0))) * 0.5;
}

static int flatten_exact(MfxScene *s)
{
    if (s->x_ready) return MFX_OK;
    const int n = (int)s->prims.size();
    std::vector<NodeX> nodes(s->nodes.size());
    for (size_t i = 0; i < nodes.size(); i++) {
        memset(&nodes[i], 0, sizeof(NodeX));
        for (int a = 0; a < 3; a++) { nodes[i].pmin[a] = s->nodes[i].pmin[a]; nodes[i].pmax[a] = s->nodes[i].pmax[a]; }
        nodes[i].first = s->nodes[i].first; nodes[i].count = s->nodes[i].count;
        if (s->integrator == MFX_SKY_TRACER) {
            // ListHit tests no boxes (RayTracing.fs:256-258): the tree must only ever skip spheres the formula would
            // reject, so every box is padded far beyond the rounding of `center -+ radius` and of the slab divisions
            for (int a = 0; a < 3; a++) {
                const double pad = 1e-7 * std::max(1.0, std::max(std::fabs(nodes[i].pmin[a]), std::fabs(nodes[i].pmax[a])));
                nodes[i].pmin[a] -= pad; nodes[i].pmax[a] += pad;
            }
        }
    }
    std::vector<PrimX> prims(n);
    std::vector<int> ref(n);
    for (int slot = 0; slot < n; slot++) {
        const MfxPrim &p = s->prims[s->indices[slot]];
        PrimX &x = prims[slot];
        memset(&x, 0, sizeof(PrimX));
        x.kind = p.kind; x.material = p.material; ref[slot] = s->indices[slot];
        if (p.kind == MFX_SPHERE) { hst(x.v0, hld(p.v)); x.e1[0] = p.v[3]; }
        else {
            H3 v0 = hld(p.v), v1 = hld(p.v + 3), v2 = hld(p.v + 6);
            hst(x.v0, v0); hst(x.e1, hsub(v1, v0)); hst(x.e2, hsub(v2, v0));
            if (p.kind == MFX_RECT) hst(x.e3, hsub(hld(p.v + 9), v0));
        }
    }
    std::vector<MatX> mats(s->mats.size());
    for (size_t i = 0; i < mats.size(); i++) {
        mats[i].kind = s->mats[i].kind; mats[i].pad = 0;
        for (int a = 0; a < 3; a++) mats[i].albedo[a] = s->mats[i].albedo[a];
        mats[i].fuzz = s->mats[i].fuzz; mats[i].ei = s->mats[i].ei; mats[i].et = s->mats[i].et;
    }
    NodeX *dn; PrimX *dp; int *dr; MatX *dm;
    MFX_TRY(upload(s, &dn, nodes)); MFX_TRY(upload(s, &dp, prims)); MFX_TRY(upload(s, &dr, ref)); MFX_TRY(upload(s, &dm, mats));
    s->x_bytes = nodes.size() * sizeof(NodeX) + prims.size() * sizeof(PrimX) + ref.size() * 4 + mats.size() * sizeof(MatX);
    SceneX &sx = s->sx;
    memset(&sx, 0, sizeof(sx));
    sx.nodes = dn; sx.prims = dp; sx.ref_id = dr; sx.mats = dm;
    const double *lp = s->light.p;
    H3 p0 = hld(lp), p1 = hld(lp + 3), p2 = hld(lp + 6), p3 = hld(lp + 9);
    tri_sample_x(sx.light.t1, p0, p1, p2);                      // Rect(p0,p1,p2,p3,0), Light.fs:38 / Rect.fs:17-19
    tri_sample_x(sx.light.t2, p0, p2, p3);
    sx.light.area = tri_area(p0, p1, p2) + tri_area(p0, p2, p3);   // Rect.fs:24
    for (int a = 0; a < 3; a++) { sx.light.normal[a] = s->light.normal[a]; sx.light.color[a] = s->light.color[a]; }
    memcpy(sx.cam.pos, s->camera.pos, 24); memcpy(sx.cam.topleft, s->camera.topleft, 24);
    memcpy(sx.cam.right, s->camera.right, 24); memcpy(sx.cam.down, s->camera.down, 24);
    memcpy(sx.lens.u, s->lens.u, 24); memcpy(sx.lens.v, s->lens.v, 24); sx.lens.radius = s->lens.lens_radius;
    if (!s->perlin_rf.empty() && !s->perlin_perm.empty()) {
        double *drf; int *dpm;
        std::vector<int> pm(s->perlin_perm.begin(), s->perlin_perm.end());
        MFX_TRY(upload(s, &drf, s->perlin_rf)); MFX_TRY(upload(s, &dpm, pm));
        sx.perlin_rf = drf; sx.perlin_perm = dpm;
    }
    sx.width = s->width; sx.height = s->height; sx.max_depth = s->max_depth; sx.mode = s->integrator; sx.n_prims = n;
    s->x_ready = true;
    return MFX_OK;
}

// ---- flatten: fast layout
static float round_down(double x)
{
    float f = (float)x;
    if ((double)f > x) f = std::nextafterf(f, -INFINITY);
    return f;
}
static float round_up(double x)
{
    float f = (float)x;
    if ((double)f < x) f = std::nextafterf(f, INFINITY);
    return f;
}
static float int_bits(int v) { float f; memcpy(&f, &v, 4); return f; }

// Materials, light, camera and frame constants shared by both fast layouts.
static int fill_fast_common(MfxScene *s, SceneF &sf)
{
    if (!s->d_matf) {
        std::vector<MatF> mats(s->mats.size());
        for (size_t i = 0; i < mats.size(); i++) {
            for (int a = 0; a < 3; a++) mats[i].albedo[a] = (float)s->mats[i].albedo[a];
            mats[i].kind = s->mats[i].kind; mats[i].fuzz = (float)s->mats[i].fuzz;
            mats[i].ei = (float)s->mats[i].ei; mats[i].et = (float)s->mats[i].et; mats[i].pad = 0.f;
        }
        MFX_TRY(upload(s, &s->d_matf, mats));
    }
    sf.mats = s->d_matf;
    const double *lp = s->light.p;
    H3 p0 = hld(lp), p1 = hld(lp + 3), p2 = hld(lp + 6), p3 = hld(lp + 9);
    H3 e;
    for (int a = 0; a < 3; a++) { sf.light.v0a[a] = (float)lp[a]; sf.light.v0b[a] = (float)lp[a]; }
    e = hsub(p1, p0); sf.light.e1a[0] = (float)e.x; sf.light.e1a[1] = (float)e.y; sf.light.e1a[2] = (float)e.z;
    e = hsub(p2, p0); sf.light.e2a[0] = (float)e.x; sf.light.e2a[1] = (float)e.y; sf.light.e2a[2] = (float)e.z;
    sf.light.e1b[0] = (float)e.x; sf.light.e1b[1] = (float)e.y; sf.light.e1b[2] = (float)e.z;
    e = hsub(p3, p0); sf.light.e2b[0] = (float)e.x; sf.light.e2b[1] = (float)e.y; sf.light.e2b[2] = (float)e.z;
    const double area = tri_area(p0, p1, p2) + tri_area(p0, p2, p3);
    sf.light.area = (float)area; sf.light.inv_pdf = (float)area;
    for (int a = 0; a < 3; a++) { sf.light.normal[a] = (float)s->light.normal[a]; sf.light.color[a] = (float)s->light.color[a]; }
    for (int a = 0; a < 3; a++) {
        sf.cam.pos[a] = (float)s->camera.pos[a]; sf.cam.topleft[a] = (float)s->camera.topleft[a];
        sf.cam.right[a] = (float)s->camera.right[a]; sf.cam.down[a] = (float)s->camera.down[a];
    }
    memcpy(sf.camx.pos, s->camera.pos, 24); memcpy(sf.camx.topleft, s->camera.topleft, 24);
    memcpy(sf.camx.right, s->camera.right, 24); memcpy(sf.camx.down, s->camera.down, 24);
    memcpy(sf.lens.u, s->lens.u, 24); memcpy(sf.lens.v, s->lens.v, 24); sf.lens.radius = s->lens.lens_radius;
    if (!s->perlin_rf.empty() && !s->perlin_perm.empty()) {
        if (!s->d_perlin_rf) {
            std::vector<float> rf(s->perlin_rf.begin(), s->perlin_rf.end());
            std::vector<int> pm(s->perlin_perm.begin(), s->perlin_perm.end());
            MFX_TRY(upload(s, &s->d_perlin_rf, rf)); MFX_TRY(upload(s, &s->d_perlin_perm, pm));
        }
        sf.perlin_rf = s->d_perlin_rf; sf.perlin_perm = s->d_perlin_perm;
    }
    sf.width = s->width; sf.height = s->height; sf.max_depth = s->max_depth; sf.mode = s->integrator;
    sf.n_mats = (int)s->mats.size();
    return MFX_OK;
}

// Fast slots of one primitive: a Rect becomes its two triangles (Rect.fs:17-19).  `id` (< 2^30) is what a ray that
// starts on the primitive carries to avoid re-hitting it; bit 30 of b.w tells the two halves of a Rect apart.
static void make_fast_slots(const MfxPrim &p, int id, std::vector<SlotF> &slots, std::vector<float4> &nrm, int &has_big)
{
    if (p.kind == MFX_SPHERE) {
        SlotF f; memset(&f, 0, sizeof(f));
        if (std::fabs(p.v[3]) >= 32.0) {
            has_big = 1;
            // big sphere: centre and radius kept as f64 bit pairs, solved in f64 by the kernel
            auto lo = [](double x) { uint64_t u; memcpy(&u, &x, 8); return int_bits((int)(uint32_t)u); };
            auto hi = [](double x) { uint64_t u; memcpy(&u, &x, 8); return int_bits((int)(uint32_t)(u >> 32)); };
            f.a = make_float4(lo(p.v[3]), hi(p.v[3]), 0.f, int_bits(3));
            f.b = make_float4(lo(p.v[0]), hi(p.v[0]), 0.f, int_bits(id));
            f.c = make_float4(lo(p.v[1]), hi(p.v[1]), lo(p.v[2]), hi(p.v[2]));
        } else {
            f.a = make_float4((float)p.v[0], (float)p.v[1], (float)p.v[2], int_bits(2));
            f.b = make_float4((float)p.v[3], (float)(p.v[3] * p.v[3]), 0.f, int_bits(id));
        }
        slots.push_back(f);
        nrm.push_back(make_float4(0.f, 0.f, 0.f, int_bits(p.material)));
        return;
    }
    const int ntri = (p.kind == MFX_RECT) ? 2 : 1;
    for (int k = 0; k < ntri; k++) {
        H3 v0 = hld(p.v), v1 = hld(p.v + 3 * (1 + k)), v2 = hld(p.v + 3 * (2 + k));
        H3 e1 = hsub(v1, v0), e2 = hsub(v2, v0);
        H3 a = hcross(e1, e2);
        double al = hlen(a);
        H3 nm = h3(a.x / al, a.y / al, a.z / al);       // Trangle.fs:110-112
        SlotF f; memset(&f, 0, sizeof(f));
        f.a = make_float4((float)v0.x, (float)v0.y, (float)v0.z, int_bits(0));
        f.b = make_float4((float)e1.x, (float)e1.y, (float)e1.z, int_bits(id | (k << 30)));
        f.c = make_float4((float)e2.x, (float)e2.y, (float)e2.z, 0.f);
        slots.push_back(f);
        nrm.push_back(make_float4((float)nm.x, (float)nm.y, (float)nm.z, int_bits(p.material)));
    }
}

// Reference-tree layout (children pairs indexed by the heap index): used by the instrumented counting runs (k_f_trace4:
// the roofline's record counts are defined on the reference tree) and by the exact shadow walk (k_h_shadow_x).
static int flatten_fast_ref(MfxScene *s)
{
    if (s->fr_ready) return MFX_OK;
    const int n = (int)s->prims.size();
    // fast slots in leaf order
    std::vector<SlotF> slots; std::vector<float4> nrm; std::vector<int> ffirst(n + 1), ref(n);
    int has_big = 0;
    slots.reserve(n); nrm.reserve(n);
    for (int slot = 0; slot < n; slot++) {
        ref[slot] = s->indices[slot];
        ffirst[slot] = (int)slots.size();
        make_fast_slots(s->prims[s->indices[slot]], slot, slots, nrm, has_big);
    }
    ffirst[n] = (int)slots.size();
    auto leaf_meta = [&](const MfxBvhNode &nd) {
        const int f0 = ffirst[nd.first], f1 = ffirst[nd.first + nd.count];
        return (f0 << 3) | (f1 - f0);
    };
    // children pairs, indexed by the interior node's heap index
    std::vector<PairF> pairs;
    SceneF &sf = s->sf_ref;
    memset(&sf, 0, sizeof(sf));
    const MfxBvhNode &root = s->nodes[0];
    for (int a = 0; a < 3; a++) { sf.root_min[a] = round_down(root.pmin[a]); sf.root_max[a] = round_up(root.pmax[a]); }
    sf.root_meta = -1;
    int max_interior = 0;
    if (root.count <= MFX_LEAF_NODE_COUNT) sf.root_meta = leaf_meta(root);
    else {
        std::vector<int> todo{ 0 };
        while (!todo.empty()) {
            const int i = todo.back(); todo.pop_back();
            // the record of heap node i (0-based) lives at index i+1 = its 1-based heap index h, so the
            // records of two siblings (2h, 2h+1) share one 128-byte line
            if ((size_t)i + 1 >= pairs.size()) { PairF z; memset(&z, 0, sizeof(z)); z.q3 = make_float4(int_bits(0), int_bits(0), 0.f, 0.f); pairs.resize(i + 2, z); }
            max_interior = std::max(max_interior, i);
            const MfxBvhNode &L = s->nodes[2 * i + 1], &R = s->nodes[2 * i + 2];
            const bool li = L.count > MFX_LEAF_NODE_COUNT, ri = R.count > MFX_LEAF_NODE_COUNT;
            PairF &pr = pairs[i + 1];
            pr.q0 = make_float4(round_down(L.pmin[0]), round_down(L.pmin[1]), round_down(L.pmin[2]), round_up(L.pmax[0]));
            pr.q1 = make_float4(round_up(L.pmax[1]), round_up(L.pmax[2]), round_down(R.pmin[0]), round_down(R.pmin[1]));
            pr.q2 = make_float4(round_down(R.pmin[2]), round_up(R.pmax[0]), round_up(R.pmax[1]), round_up(R.pmax[2]));
            pr.q3 = make_float4(int_bits(li ? -1 : leaf_meta(L)), int_bits(ri ? -1 : leaf_meta(R)), 0.f, 0.f);
            if (li) todo.push_back(2 * i + 1);
            if (ri) todo.push_back(2 * i + 2);
        }
    }
    PairF *dpairs; SlotF *dslots; float4 *dnrm; int *dref;
    MFX_TRY(upload(s, &dpairs, pairs)); MFX_TRY(upload(s, &dslots, slots)); MFX_TRY(upload(s, &dnrm, nrm));
    MFX_TRY(upload(s, &dref, ref));
    s->fr_bytes = pairs.size() * sizeof(PairF) + slots.size() * sizeof(SlotF) + nrm.size() * 16 + ref.size() * 4;
    sf.pairs = dpairs; sf.slots = dslots; sf.slot_nrm = dnrm; sf.ref_id = dref; sf.slot_prim = nullptr;
    MFX_TRY(fill_fast_common(s, sf));
    sf.n_slots = (int)slots.size();
    sf.has_big_sphere = has_big;
    { int depth = 0; for (unsigned v = (unsigned)max_interior + 1u; v > 1u; v >>= 1) depth++; sf.levels = depth + 2; }
    s->fr_ready = true;
    return MFX_OK;
}

// ---- flatten: fast layout over the library's own tree (mfx_build.cpp: binned SAH, collapsed to four children per record)
// The host half (slots, bounds, tree build, reordering) depends on the primitives alone, so it is cached by content:
// the replicas of a multi-GPU scene (mfx_multi_create) and a host that re-creates its Scene every frame (Scene.fs
// builds a new Bvh per `new Scene(state)`) pay for it once.  Two independent 64-bit hashes over the primitive bytes
// key the cache; a handful of entries, bounded in bytes, least recently used goes first.
struct OwnTreeHost {
    std::vector<QuadF> quads;
    std::vector<SlotF> slots;
    std::vector<float4> nrm;
    std::vector<int> slot_prim;         // own-tree fast slot -> primitive index, bit 30 = second triangle of a Rect
    int depth = 0, has_big = 0;
    size_t bytes() const { return quads.size() * sizeof(QuadF) + slots.size() * sizeof(SlotF) + nrm.size() * 16 + slot_prim.size() * 4; }
};
struct TreeKey {
    uint64_t h1, h2; size_t n; long max_leaf, trav, collapse;
    bool operator==(const TreeKey &o) const { return h1 == o.h1 && h2 == o.h2 && n == o.n && max_leaf == o.max_leaf && trav == o.trav && collapse == o.collapse; }
};
static std::mutex g_tree_mu;
static std::vector<std::pair<TreeKey, std::shared_ptr<OwnTreeHost>>> g_tree_cache;    // most recently used last
static const size_t TREE_CACHE_BYTES = (size_t)6 << 30, TREE_CACHE_ENTRIES = 8;

static TreeKey tree_key(const std::vector<MfxPrim> &prims, long max_leaf, long trav)
{
    const uint64_t *w = reinterpret_cast<const uint64_t *>(prims.data());
    const size_t nw = prims.size() * sizeof(MfxPrim) / 8;
    uint64_t a = 0x9E3779B97F4A7C15ull, b = 0xC2B2AE3D27D4EB4Full;
    for (size_t i = 0; i < nw; i++) {
        a = (a ^ w[i]) * 0x100000001B3ull; a ^= a >> 29;
        b = (b + w[i]) * 0xFF51AFD7ED558CCDull; b ^= b >> 32;
    }
    return TreeKey{ a, b, prims.size(), max_leaf, trav, env_long("MFX_COLLAPSE_DP", 100) * 1000 + env_long("MFX_TREE_OPT", 2) };     // (every builder knob that shapes the tree)
}

static std::shared_ptr<OwnTreeHost> build_own_tree_host(MfxScene *s, long max_leaf, long trav)
{
    const auto t_begin = std::chrono::steady_clock::now();
    auto lap = [&](const char *what) {
        if (env_long("MFX_DEBUG", 0))
            fprintf(stderr, "[mfx] flatten_fast %-10s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count());
    };
    auto out = std::make_shared<OwnTreeHost>();
    const int n = (int)s->prims.size();
    std::vector<SlotF> raw; std::vector<float4> raw_nrm;
    int has_big = 0;
    raw.reserve(n); raw_nrm.reserve(n);
    std::vector<int> owner;                                     // raw slot -> primitive
    owner.reserve(n);
    for (int i = 0; i < n; i++) {
        const size_t before = raw.size();
        make_fast_slots(s->prims[i], i, raw, raw_nrm, has_big);
        for (size_t k = before; k < raw.size(); k++) owner.push_back(i);
    }
    const int ns = (int)raw.size();
    // slot bounds, rounded outward from the f64 vertices
    std::vector<float> blo((size_t)ns * 3), bhi((size_t)ns * 3);
    for (int k = 0; k < ns; k++) {
        const MfxPrim &p = s->prims[owner[k]];
        double lo[3], hi[3];
        if (p.kind == MFX_SPHERE) {
            for (int a = 0; a < 3; a++) { lo[a] = p.v[a] - std::fabs(p.v[3]); hi[a] = p.v[a] + std::fabs(p.v[3]); }
        } else {
            const int sub = (p.kind == MFX_RECT && k > 0 && owner[k - 1] == owner[k]) ? 1 : 0;
            const double *v[3] = { p.v, p.v + 3 * (1 + sub), p.v + 3 * (2 + sub) };
            for (int a = 0; a < 3; a++) { lo[a] = std::min(v[0][a], std::min(v[1][a], v[2][a])); hi[a] = std::max(v[0][a], std::max(v[1][a], v[2][a])); }
        }
        for (int a = 0; a < 3; a++) { blo[(size_t)k * 3 + a] = round_down(lo[a]); bhi[(size_t)k * 3 + a] = round_up(hi[a]); }
    }
    lap("slots");
    MfxOwnTree tree;
    // The builder forks its top levels over threads (identical tree for any fork depth).  One process per GPU means
    // `world` builders on one host at the same time: eight of them forking 32 ways each on a 16-thread host take longer
    // than eight serial ones, so the fork depth follows the threads this rank can expect for itself.
    int par_depth = 0;
    for (unsigned share = std::max(1u, std::thread::hardware_concurrency()) / (unsigned)std::max(1, s->host_share); share > 1 && par_depth < 5; share >>= 1) par_depth++;
    par_depth = (int)env_long("MFX_BVH_BUILD_PAR_DEPTH", par_depth);
    mfx_build_own_tree(blo.data(), bhi.data(), ns, (int)max_leaf, (float)trav * 0.01f, par_depth, tree);
    lap("own tree");
    const std::vector<int> &order = tree.order;
    out->depth = tree.depth; out->has_big = has_big;
    out->slots.resize(ns); out->nrm.resize(ns); out->slot_prim.resize(ns);
    for (int k = 0; k < ns; k++) {      // bit 30: the second triangle of a Rect (raw slots of one primitive are adjacent)
        const int raw_k = order[k];
        out->slots[k] = raw[raw_k]; out->nrm[k] = raw_nrm[raw_k];
        out->slot_prim[k] = owner[raw_k] | ((raw_k > 0 && owner[raw_k - 1] == owner[raw_k]) ? (1 << 30) : 0);
    }
    out->quads = std::move(tree.quads);
    lap("reorder");
    return out;
}

static int flatten_fast(MfxScene *s)
{
    if (s->f_ready) return MFX_OK;
    if (s->prims.size() > ((size_t)1 << 27)) return fail(MFX_ERR_INVALID_ARGUMENT, "too many primitives (%zu)", s->prims.size());
    const long max_leaf = std::min(7L, std::max(1L, env_long("MFX_SAH_MAX_LEAF", 4))), trav = env_long("MFX_SAH_TRAV_COST_PCT", 100);
    std::shared_ptr<OwnTreeHost> host;
    {
        const TreeKey key = tree_key(s->prims, max_leaf, trav);      // hashed outside the lock: replicas hash side by side
        // one builder at a time: the replicas of one scene arrive together, the first one builds, the others find it
        std::lock_guard<std::mutex> g(g_tree_mu);
        const bool use_cache = env_long("MFX_TREE_CACHE", 1) != 0;
        for (size_t i = 0; use_cache && i < g_tree_cache.size(); i++)
            if (g_tree_cache[i].first == key) {
                host = g_tree_cache[i].second;
                std::rotate(g_tree_cache.begin() + (long)i, g_tree_cache.begin() + (long)i + 1, g_tree_cache.end());
                break;
            }
        if (!host) {
            host = build_own_tree_host(s, max_leaf, trav);
            if (use_cache && host->bytes() <= TREE_CACHE_BYTES) {
                g_tree_cache.push_back({ key, host });
                size_t total = 0;
                for (auto &e : g_tree_cache) total += e.second->bytes();
                while (g_tree_cache.size() > TREE_CACHE_ENTRIES || total > TREE_CACHE_BYTES) { total -= g_tree_cache.front().second->bytes(); g_tree_cache.erase(g_tree_cache.begin()); }
            }
        }
    }
    const std::vector<QuadF> &quads = host->quads;
    const int ns = (int)host->slots.size();
    s->f_slot_prim = host->slot_prim;

    SceneF &sf = s->sf;
    memset(&sf, 0, sizeof(sf));
    SlotF *dslots; float4 *dnrm; QuadF *dquads;
    MFX_TRY(upload(s, &dquads, quads)); MFX_TRY(upload(s, &dslots, host->slots)); MFX_TRY(upload(s, &dnrm, host->nrm));
    s->own_host = host;
    s->f_bytes = quads.size() * sizeof(QuadF) + host->slots.size() * sizeof(SlotF) + host->nrm.size() * 16 + s->mats.size() * sizeof(MatF);
    sf.quads = dquads; sf.slots = dslots; sf.slot_nrm = dnrm;
    sf.ref_id = nullptr;                                        // b.w already holds the caller's primitive index
    sf.root_meta = -1;
    sf.own_tree = 1; sf.own_depth = host->depth;
    sf.stack_smem = (int)std::min((long)std::min(3 * host->depth, MFX_STACK_SMEM_MAX), std::max(1L, env_long("MFX_STACK_SMEM", 12)));
    sf.spill_threads = s->sm_count * 16 * 128;                  // most threads a persistent 128-thread grid can hold
    if (const size_t spill = own_spill_entries(sf)) {
        MFX_TRY(dev_alloc_t(s, &sf.stack_spill, spill));
        s->f_bytes += spill * sizeof(uint2);
    }
    MFX_TRY(fill_fast_common(s, sf));
    sf.n_slots = ns;
    sf.n_quads = (int)quads.size();
    sf.has_big_sphere = host->has_big;
    s->f_ready = true;
    return MFX_OK;
}

// Which fast layout a call runs on: the own tree, unless the caller asked for traversal counters (defined on the
// reference tree).
static int fast_layout(MfxScene *s, bool counting, const SceneF **out)
{
    if (counting) { MFX_TRY(flatten_fast_ref(s)); *out = &s->sf_ref; }
    else { MFX_TRY(flatten_fast(s)); *out = &s->sf; }
    return MFX_OK;
}

// ---- flatten: the tables of the id-exact hybrid traversal (mfx_hybrid.cu) on top of the exact and the own-tree layouts
static int flatten_hybrid(MfxScene *s)
{
    if (s->h_ready) return MFX_OK;
    MFX_TRY(flatten_exact(s)); MFX_TRY(flatten_fast(s));
    const int n = (int)s->prims.size(), ns = (int)s->f_slot_prim.size();
    std::vector<int> ref_of_prim(n), leaf_of_ref(n, 0);
    std::vector<PrimH> ph(ns);
    std::vector<int2> ref_fslot(n, make_int2(-1, -1));
    for (int slot = 0; slot < n; slot++) ref_of_prim[s->indices[slot]] = slot;
    for (int k = 0; k < ns; k++) {
        const int prim = s->f_slot_prim[k] & 0x3fffffff, half = s->f_slot_prim[k] >> 30;
        const int ref = ref_of_prim[prim];
        if (half) ref_fslot[ref].y = k; else ref_fslot[ref].x = k;
        const MfxPrim &p = s->prims[prim];
        PrimH &x = ph[k];
        memset(&x, 0, sizeof(PrimH));
        x.ref = ref;
        if (p.kind == MFX_SPHERE) { x.kind = 2; hst(x.v0, hld(p.v)); x.e1[0] = p.v[3]; }
        else {      // the same subtractions as flatten_exact: bit-identical edge vectors
            H3 v0 = hld(p.v), v1 = hld(p.v + 3), v2 = hld(p.v + 6);
            hst(x.v0, v0); hst(x.e1, hsub(v1, v0)); hst(x.e2, hsub(v2, v0));
            x.kind = half ? 1 : 0;
            if (p.kind == MFX_RECT) hst(x.e3, hsub(hld(p.v + 9), v0));
        }
    }
    // reference tree: depth-first walk from the root, leaf iff count <= LeafNodeCount (BvhNode.fs:39,44)
    {
        std::vector<int> todo{ 0 };
        while (!todo.empty()) {
            const int i = todo.back(); todo.pop_back();
            const MfxBvhNode &nd = s->nodes[i];
            if (nd.count > MFX_LEAF_NODE_COUNT) { todo.push_back(2 * i + 2); todo.push_back(2 * i + 1); continue; }
            for (int k = 0; k < nd.count; k++) leaf_of_ref[nd.first + k] = i;
        }
    }
    SceneH &sh = s->sh;
    memset(&sh, 0, sizeof(sh));
    int *d_leaf; int2 *d_fslot; PrimH *d_ph;
    MFX_TRY(upload(s, &d_ph, ph)); MFX_TRY(upload(s, &d_leaf, leaf_of_ref)); MFX_TRY(upload(s, &d_fslot, ref_fslot));
    sh.prims_h = d_ph; sh.leaf_of_ref = d_leaf; sh.ref_fslot = d_fslot;
    double m = 0.;
    for (int a = 0; a < 3; a++) m = std::max(m, std::max(std::fabs(s->nodes[0].pmin[a]), std::fabs(s->nodes[0].pmax[a])));
    sh.max_abs = round_up(m);
    sh.n_ref = n;
    sh.pad_factor = (float)env_long("MFX_HYB_PAD_PPB", 4000) * 1e-9f;
    s->h_bytes = (uint64_t)ns * sizeof(PrimH) + (uint64_t)n * 12;
    s->h_ready = true;
    return MFX_OK;
}

// the hybrid's per-wave buffers follow the fast wave's capacity (they are only allocated once the hybrid is used)
static int ensure_wave_hybrid(MfxScene *s)
{
    if (s->wh_ready && s->wh_P == s->wf.P) return MFX_OK;
    WaveH &w = s->wh;
    if (s->wh_ready) {
        CUDA_TRY(cudaStreamSynchronize(s->stream));
        void *old[] = { w.dir64, w.org64, w.t, w.ref, w.fix_q, w.fix_n };
        for (void *q : old) dev_free_one(s, q);
        s->wh_ready = false;
    }
    memset(&w, 0, sizeof(w));
    const size_t P = (size_t)s->wf.P;
    MFX_TRY(dev_alloc_t(s, &w.dir64, 3 * P)); MFX_TRY(dev_alloc_t(s, &w.org64, 3 * P)); MFX_TRY(dev_alloc_t(s, &w.t, P)); MFX_TRY(dev_alloc_t(s, &w.ref, P));
    MFX_TRY(dev_alloc_t(s, &w.fix_q, (size_t)MFX_HYB_FIX_CAP)); MFX_TRY(dev_alloc_t(s, &w.fix_n, 4));
    s->wh_P = (int)P; s->wh_ready = true;
    return MFX_OK;
}

static bool use_hybrid(int flags);
static int ensure_frame_buffers(MfxScene *s);

// Builds the device layouts a Sample of this precision will use (exact: reference tree + f64 primitives; fast: own SAH tree,
// f32 slots and the id-exact tables) now instead of inside the first Sample: a host that pipelines frames does it while the
// previous frame renders.
extern "C" int mfx_scene_prepare(MfxScene *s, int32_t precision)
{
    if (!s) return fail(MFX_ERR_INVALID_ARGUMENT, "null scene");
    if (precision != MFX_EXACT_F64 && precision != MFX_FAST_F32) return fail(MFX_ERR_INVALID_ARGUMENT, "unknown precision %d", precision);
    MFX_TRY(bind_device(s->device));
    if (precision == MFX_EXACT_F64) MFX_TRY(flatten_exact(s));
    else {
        MFX_TRY(flatten_fast(s));
        if (use_hybrid(0)) MFX_TRY(flatten_hybrid(s));
    }
    MFX_TRY(ensure_frame_buffers(s));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return MFX_OK;
}

extern "C" int mfx_scene_device_bytes(const MfxScene *sc, uint64_t *exact_bytes, uint64_t *fast_bytes)
{
    if (!sc) return fail(MFX_ERR_INVALID_ARGUMENT, "null scene");
    MfxScene *s = const_cast<MfxScene *>(sc);
    MFX_TRY(bind_device(s->device));
    MFX_TRY(flatten_exact(s)); MFX_TRY(flatten_fast(s));
    if (exact_bytes) *exact_bytes = s->x_bytes;
    if (fast_bytes) *fast_bytes = s->f_bytes;
    return MFX_OK;
}

// ---- per-wave path state
static int ensure_wave_exact(MfxScene *s)
{
    if (s->wx_ready) return MFX_OK;
    const size_t P = (size_t)env_long("MFX_WAVE_PATHS_EXACT", 1 << 20);
    const size_t V = (size_t)s->max_depth + 1;
    WaveX &w = s->wx;
    memset(&w, 0, sizeof(w));
    w.P = (int)P;
    MFX_TRY(dev_alloc_t(s, &w.ray_o, 3 * P)); MFX_TRY(dev_alloc_t(s, &w.ray_d, 3 * P));
    MFX_TRY(dev_alloc_t(s, &w.hit_t, P)); MFX_TRY(dev_alloc_t(s, &w.hit_slot, P));
    MFX_TRY(dev_alloc_t(s, &w.sh_d, 3 * P)); MFX_TRY(dev_alloc_t(s, &w.sh_dist, P));
    const bool sky = (s->integrator == MFX_SKY_TRACER);      // keeps one terminal colour and the attenuations only
    MFX_TRY(dev_alloc_t(s, &w.v_l, (sky ? 1 : V) * 3 * P)); MFX_TRY(dev_alloc_t(s, &w.v_col, V * 3 * P));
    MFX_TRY(dev_alloc_t(s, &w.v_ei, (sky ? 1 : V) * P)); MFX_TRY(dev_alloc_t(s, &w.v_kind, (sky ? 1 : V) * P));
    MFX_TRY(dev_alloc_t(s, &w.nv, P));
    MFX_TRY(dev_alloc_t(s, &w.queue[0], P)); MFX_TRY(dev_alloc_t(s, &w.queue[1], P));
    MFX_TRY(dev_alloc_t(s, &w.counts, MFX_COUNTS_LEN));
    s->wx_ready = true;
    return MFX_OK;
}

// Path state of one wave, fast precision.  Bigger waves mean fewer, longer launches: on C2 a 4 Mi-path wave (2 spp of
// 1080p) costs 25 % against 32-64 Mi because every persistent launch pays its ramp-up and its tail (profiles/), so
// the wave is sized for the call at hand -- pixels x spp -- up to MFX_WAVE_PATHS (default 128 Mi paths = 24.6 GB of
// the 180 GB) and only ever grows.
static int ensure_wave_fast(MfxScene *s, size_t want, bool at_least = false)
{
    // at_least: the caller needs room for `want` entries whatever the cap says (the exact wavefront borrows these queues)
    const size_t cap = at_least ? want : (size_t)std::max(1024L, env_long("MFX_WAVE_PATHS", 1L << 27));
    size_t P = std::min(cap, std::max(want, (size_t)1 << 16));
    if (at_least) P = std::max(want, (size_t)1 << 16);
    if (s->wf_ready && (size_t)s->wf.P >= P) return MFX_OK;
    WaveF &w = s->wf;
    if (s->wf_ready) {
        CUDA_TRY(cudaStreamSynchronize(s->stream));
        void *old[] = { w.ray_o[0], w.ray_o[1], w.ray_d[0], w.ray_d[1], w.thr[0], w.thr[1], w.hit, w.rad, w.sh_o, w.sh_d, w.sh_c, w.counts, w.dbg_stamp };
        for (void *q : old) dev_free_one(s, q);
        s->wf_ready = false;
    }
    // a wave that does not fit (another tenant on the GPU) is halved until it does: same frame, more launches
    bool trimmed = false;
    for (;;) {
        memset(&w, 0, sizeof(w));
        w.P = (int)P;
        w.tmin = (s->integrator == MFX_SKY_TRACER) ? (float)MFX_SKY_TMIN : 1e-6f;
        w.tmax = (s->integrator == MFX_SKY_TRACER) ? (float)MFX_SKY_TMAX : 99999999.f;
        auto all = [&]() -> int {
            for (int b = 0; b < 2; b++) {
                MFX_TRY(dev_alloc_t(s, &w.ray_o[b], P)); MFX_TRY(dev_alloc_t(s, &w.ray_d[b], P)); MFX_TRY(dev_alloc_t(s, &w.thr[b], P));
            }
            MFX_TRY(dev_alloc_t(s, &w.hit, P)); MFX_TRY(dev_alloc_t(s, &w.rad, P));
            MFX_TRY(dev_alloc_t(s, &w.sh_o, P)); MFX_TRY(dev_alloc_t(s, &w.sh_d, P)); MFX_TRY(dev_alloc_t(s, &w.sh_c, P));
            MFX_TRY(dev_alloc_t(s, &w.counts, MFX_COUNTS_LEN));
#ifdef MFX_DEBUG_CHECKS
            MFX_TRY(dev_alloc_t(s, &w.dbg_stamp, P));
            CUDA_TRY(cudaMemsetAsync(w.dbg_stamp, 0, P * sizeof(int), s->stream));
#endif
            return MFX_OK;
        };
        const int rc = all();
        if (rc == MFX_OK) break;
        void *part[] = { w.ray_o[0], w.ray_o[1], w.ray_d[0], w.ray_d[1], w.thr[0], w.thr[1], w.hit, w.rad, w.sh_o, w.sh_d, w.sh_c, w.counts, w.dbg_stamp };
        for (void *q : part) dev_free_one(s, q, false);
        if (rc != MFX_ERR_OUT_OF_MEMORY || P <= ((size_t)1 << 20)) return rc;
        cudaGetLastError();                                       // clear the allocation error
        if (!trimmed) { pool_trim(s->device); trimmed = true; } else P /= 2;
    }
    s->wf_ready = true;
    return MFX_OK;
}

static int ensure_frame_buffers(MfxScene *s)
{
    const size_t npx = (size_t)s->width * s->height;
    if (!s->d_pixsum) MFX_TRY(dev_alloc_t(s, &s->d_pixsum, 4 * npx));
    if (!s->d_color_wh) MFX_TRY(dev_alloc_t(s, &s->d_color_wh, 4 * npx));
    if (!s->d_rgba) MFX_TRY(dev_alloc_t(s, &s->d_rgba, npx));
    return MFX_OK;
}

// Interleaved square tiles: tile k (row-major over the tile grid) belongs to rank k % world.
static void tile_pixels(int width, int height, int tile, int rank, int world, std::vector<int> &pix)
{
    const int tx = (width + tile - 1) / tile, ty = (height + tile - 1) / tile;
    // sized once and filled row by row: a host that rebuilds its Scene per frame pays this per frame (1 M ids at 2 GPUs)
    size_t total = 0;
    for (int t = rank; t < tx * ty; t += world) {
        const int x0 = (t % tx) * tile, y0 = (t / tx) * tile;
        total += (size_t)(std::min(x0 + tile, width) - x0) * (size_t)(std::min(y0 + tile, height) - y0);
    }
    const size_t base = pix.size();
    pix.resize(base + total);
    int *out = pix.data() + base;
    for (int t = rank; t < tx * ty; t += world) {
        const int x0 = (t % tx) * tile, y0 = (t / tx) * tile;
        const int x1 = std::min(x0 + tile, width), y1 = std::min(y0 + tile, height);
        for (int y = y0; y < y1; y++) {
            const int row = y * width;
            for (int x = x0; x < x1; x++) *out++ = row + x;
        }
    }
}

extern "C" int mfx_tile_map(int32_t width, int32_t height, int32_t tile_size, int32_t rank, int32_t world,
                            int32_t *pixels_out, int32_t *n_out)
{
    if (width <= 0 || height <= 0 || tile_size <= 0 || world <= 0 || rank < 0 || rank >= world || !n_out)
        return fail(MFX_ERR_INVALID_ARGUMENT, "mfx_tile_map: bad arguments (w=%d h=%d tile=%d rank=%d world=%d)", width, height, tile_size, rank, world);
    std::vector<int> pix;
    tile_pixels(width, height, tile_size, rank, world, pix);
    *n_out = (int32_t)pix.size();
    if (pixels_out) memcpy(pixels_out, pix.data(), pix.size() * sizeof(int));
    return MFX_OK;
}

// pixels of rank `rank` under column-stripe ownership (TileMap)
static int stripe_pixels(int width, int height, int stripe, int rank, int world)
{
    long n = 0;
    for (int x0 = rank * stripe; x0 < width; x0 += world * stripe) n += (long)std::min(stripe, width - x0) * height;
    return (int)n;
}

// The pixels of `rank`'s column stripes out of `world`; world 1 = the whole frame (pixel_of's identity).
static TileMap stripe_tilemap(int width, int height, int stripe, int rank, int world)
{
    TileMap tm;
    memset(&tm, 0, sizeof(tm));
    tm.height = height;
    if (world <= 1) { tm.n_pix = width * height; return tm; }
    tm.stripe = stripe; tm.rank = rank; tm.world = world;
    tm.n_pix = stripe_pixels(width, height, stripe, rank, world);
    return tm;
}

// The stripe rule as a table (same local order as pixel_of computes on the device): for hosts and tests.
extern "C" int mfx_stripe_map(int32_t width, int32_t height, int32_t stripe, int32_t rank, int32_t world,
                              int32_t *pixels_out, int32_t *n_out)
{
    if (width <= 0 || height <= 0 || stripe <= 0 || world <= 0 || rank < 0 || rank >= world || !n_out)
        return fail(MFX_ERR_INVALID_ARGUMENT, "mfx_stripe_map: bad arguments (w=%d h=%d stripe=%d rank=%d world=%d)", width, height, stripe, rank, world);
    *n_out = stripe_pixels(width, height, stripe, rank, world);
    if (pixels_out) {
        int32_t *out = pixels_out;
        for (int x0 = rank * stripe; x0 < width; x0 += world * stripe) {
            const int wl = std::min(stripe, width - x0);
            for (int y = 0; y < height; y++)
                for (int x = x0; x < x0 + wl; x++) *out++ = y * width + x;
        }
    }
    return MFX_OK;
}

static int get_tilemap(MfxScene *s, int tile, int rank, int world, bool stripes, TileMap *tm)
{
    memset(tm, 0, sizeof(*tm));
    tm->height = s->height;
    if (world <= 1 || tile <= 0) {
        // one device, whole frame: path ids walk the frame in column stripes of MFX_PIXEL_STRIPE pixels (rows of 8 inside a
        // stripe), so the 32 rays a warp picks up together come from an 8 x 4 block of pixels instead of a 32 x 1 run
        const long ps = env_long("MFX_PIXEL_STRIPE", 8);
        tm->pix = nullptr; tm->n_pix = s->width * s->height;
        if (ps > 0) { tm->stripe = (int)ps; tm->rank = 0; tm->world = 1; }
        return MFX_OK;
    }
    if (stripes) {
        *tm = stripe_tilemap(s->width, s->height, tile, rank, world);
        return MFX_OK;
    }
    auto key = std::make_tuple(tile, rank, world);
    auto it = s->tilemaps.find(key);
    if (it == s->tilemaps.end()) {
        std::vector<int> pix;
        tile_pixels(s->width, s->height, tile, rank, world, pix);
        int *d = nullptr;
        MFX_TRY(upload(s, &d, pix));
        it = s->tilemaps.emplace(key, std::make_pair(d, (int)pix.size())).first;
    }
    tm->pix = it->second.first; tm->n_pix = it->second.second;
    return MFX_OK;
}

static int get_event(FrameJob &j, size_t idx, cudaEvent_t *e)
{
    while (j.events.size() <= idx) {
        cudaEvent_t ev;
        MFX_TRY(event_get(j.device, true, &ev));
        j.events.push_back(ev);
    }
    *e = j.events[idx];
    return MFX_OK;
}

// Pinned 256-byte blocks for the per-frame statistics, recycled for the life of the process: cudaMallocHost and
// cudaFreeHost synchronise the device, which a host that re-creates its Scene every frame would pay per frame.
static std::vector<void *> g_stat_blocks;
static int stat_block_get(void **p)
{
    {
        std::lock_guard<std::mutex> g(g_pool_mu);
        if (!g_stat_blocks.empty()) { *p = g_stat_blocks.back(); g_stat_blocks.pop_back(); return MFX_OK; }
    }
    CUDA_TRY(cudaHostAlloc(p, 256, cudaHostAllocPortable));
    return MFX_OK;
}
static void stat_block_put(void *p)
{
    if (!p) return;
    std::lock_guard<std::mutex> g(g_pool_mu);
    g_stat_blocks.push_back(p);
}

static int ensure_job(MfxScene *s, FrameJob &j)
{
    if (!j.d_totals) MFX_TRY(dev_alloc_t(s, &j.d_totals, 8));
    if (!j.d_ctr) MFX_TRY(dev_alloc_t(s, &j.d_ctr, 1));
    if (!j.h_totals) {      // one block: [0, 64) totals, [128, 176) traversal counters
        void *blk = nullptr;
        MFX_TRY(stat_block_get(&blk));
        j.h_totals = (unsigned long long *)blk;
        j.h_ctr = (TravCounters *)((char *)blk + 128);
    }
    j.device = s->device;
    if (!j.done) MFX_TRY(event_get(s->device, false, &j.done));
    if (!j.copied) MFX_TRY(event_get(s->device, false, &j.copied));
    return MFX_OK;
}

// MFX_FAST_F32 closest hits of bounce 0 and of the seams go through the id-exact hybrid traversal unless the caller
// (MFX_SAMPLE_F32_PRIMARY) or the environment (MFX_F32_PRIMARY=1, A/B runs) asks for f32 leaf tests everywhere.
static bool use_hybrid(int flags)
{
    return !(flags & MFX_SAMPLE_F32_PRIMARY) && env_long("MFX_F32_PRIMARY", 0) == 0;
}

// ------------------------------------------------------------------ the wavefront driver
// One IPixelIntegrator.Sample(n) call (Integrators.fs:160-172): every (pixel, sample) of this
// rank's tiles becomes one path; paths advance one vertex per bounce through
//   extend (closest hit) -> shade (BSDF + light sample, queue compaction) -> shadow (occlusion)
// and are resolved into per-pixel sums.  No host synchronisation inside: queue sizes stay on
// the device and every kernel is a persistent grid-stride loop over `counts[bounce]`.
static int finish_sample(MfxScene *s, FrameJob &job);
static int finish_oldest(MfxScene *s);

// Enqueues one Sample call on the scene's stream and returns without waiting for it.
// Frames of DIFFERENT scenes on one device render one after the other, not side by side: the kernels of a frame wait for
// the last kernel of the frame launched before it on that device (frames of one scene share a stream and are ordered
// anyway).  A host that re-creates its scene per frame and keeps two frames in flight still overlaps everything but the
// kernels -- scene creation, layout uploads, launch latency, the download -- while two persistent-grid frames side by
// side cost more than their sum: two copies of the tree compete for the L1 the traversal is bound by (measured on
// frames of 16.6 M paths, re-created scenes, two in flight: 8.35 ms per frame side by side against 7.42 alone).
// MFX_SERIALIZE_FRAMES=0 turns the ordering off.
static std::mutex g_order_mu;
static std::map<int, cudaEvent_t> g_frame_tail;

static int launch_sample(MfxScene *s, const MfxSampleParams *p, double *d_color_wh, float4 *d_rgba, FrameJob &job)
{
    if (!s || !p) return fail(MFX_ERR_INVALID_ARGUMENT, "null scene/params");
    if (p->spp <= 0) return fail(MFX_ERR_INVALID_ARGUMENT, "spp must be positive, got %d", p->spp);
    if (p->precision != MFX_EXACT_F64 && p->precision != MFX_FAST_F32) return fail(MFX_ERR_INVALID_ARGUMENT, "unknown precision %d", p->precision);
    if (p->world > 1 && (p->rank < 0 || p->rank >= p->world)) return fail(MFX_ERR_INVALID_ARGUMENT, "rank %d outside world %d", p->rank, p->world);
    if (p->world > 1 && p->tile_size <= 0) return fail(MFX_ERR_INVALID_ARGUMENT, "world > 1 needs a positive tile_size");
    MFX_TRY(bind_device(s->device));
    const bool trace_host = env_long("MFX_DEBUG", 0) >= 2;                 // host-clock anatomy of the call
    const auto th0 = std::chrono::steady_clock::now();
    auto th_ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - th0).count(); };
    const bool exact = (p->precision == MFX_EXACT_F64);
    s->host_share = s->in_process_replica ? 1 : std::max(1, p->world);
    if (exact) { MFX_TRY(flatten_exact(s)); MFX_TRY(ensure_wave_exact(s)); }
    const bool count_ref = (p->flags & MFX_SAMPLE_COUNT_TRAVERSAL) != 0;
    const bool counting = count_ref || (p->flags & MFX_SAMPLE_COUNT_OWN_TREE) != 0;
    const SceneF *sfp = nullptr;
    if (!exact) MFX_TRY(fast_layout(s, count_ref, &sfp));
    MFX_TRY(ensure_frame_buffers(s));
    TileMap tm;
    MFX_TRY(get_tilemap(s, p->tile_size, p->rank, p->world, (p->flags & MFX_SAMPLE_STRIPES) != 0, &tm));
    if (!exact) MFX_TRY(ensure_wave_fast(s, (size_t)tm.n_pix * (size_t)p->spp));
    // bounce 0 of the throughput path is traced id-exactly (mfx_hybrid.cu) unless the caller opts out
    const bool hyb = !exact && sfp->own_tree && !counting && use_hybrid(p->flags);
    if (hyb) { MFX_TRY(flatten_hybrid(s)); MFX_TRY(ensure_wave_hybrid(s)); }
    // ... and the exact precision sends ITS closest-hit queries through the same kernel (same answers as bvh_hit_x, bit for
    // bit, on the own tree instead of ~50 f64 box tests per ray on the reference's); MFX_EXACT_WALK=1 keeps the plain walk
    const bool hyb_x = exact && !counting && env_long("MFX_EXACT_WALK", 0) == 0;
    if (hyb_x) {
        MFX_TRY(flatten_hybrid(s));
        MFX_TRY(ensure_wave_fast(s, (size_t)s->wx.P, true));
        if (s->wf.P < s->wx.P) return fail(MFX_ERR_OUT_OF_MEMORY, "no room for the exact wavefront's closest-hit queue");
        MFX_TRY(ensure_wave_hybrid(s));
        if (s->integrator != MFX_SKY_TRACER) MFX_TRY(flatten_fast_ref(s));                  // the f32 copy of the reference tree: the exact shadow walk
        s->wf.cam_origin = 0;
        CUDA_TRY(cudaMemsetAsync(s->wf.counts, 0, MFX_COUNTS_LEN * sizeof(int), s->stream));
    }
    MFX_TRY(ensure_job(s, job));
    TravCounters *ctr = counting ? job.d_ctr : nullptr;
    const bool sky = (s->integrator == MFX_SKY_TRACER);
    if (!exact) s->wf.cam_origin = (sfp->own_tree && !counting && !(sky && s->lens.lens_radius != 0.0)) ? 1 : 0;
    const size_t npx = (size_t)s->width * s->height;
    cudaStream_t st = s->stream;
    LaunchCfg cfg{ s->sm_count, 128, st, (p->flags & MFX_SAMPLE_REFERENCE_STREAM) ? 1 : 0, 0 };

    CUDA_TRY(cudaMemsetAsync(s->d_pixsum, 0, 4 * npx * sizeof(double), st));
    CUDA_TRY(cudaMemsetAsync(job.d_totals, 0, 8 * sizeof(unsigned long long), st));
    CUDA_TRY(cudaMemsetAsync(job.d_ctr, 0, sizeof(TravCounters), st));
    if ((tm.pix || tm.stripe) && !(p->flags & MFX_SAMPLE_NO_CLEAR)) {   // pixels of other ranks must read as zero
        if (d_color_wh) CUDA_TRY(cudaMemsetAsync(d_color_wh, 0, 4 * npx * sizeof(double), st));
        if (d_rgba) CUDA_TRY(cudaMemsetAsync(d_rgba, 0, npx * sizeof(float4), st));
    }
    const double th_prepared = th_ms();
    size_t ev = 0;
    cudaEvent_t e_begin, e_end;
    MFX_TRY(get_event(job, ev++, &e_begin)); MFX_TRY(get_event(job, ev++, &e_end));
    job.e_begin = 0; job.e_end = 1;
    const bool ordered = env_long("MFX_SERIALIZE_FRAMES", 1) != 0;
    if (ordered) {
        std::lock_guard<std::mutex> g(g_order_mu);
        auto it = g_frame_tail.find(s->device);
        if (it != g_frame_tail.end()) CUDA_TRY(cudaStreamWaitEvent(st, it->second, 0));
    }
    CUDA_TRY(cudaEventRecord(e_begin, st));
    std::vector<Span> &spans = job.spans;
    spans.clear();
    auto timed = [&](int cls, cudaStream_t on) -> int {      // returns via spans the event pair bracketing the next launch
        cudaEvent_t a, b;
        MFX_TRY(get_event(job, ev, &a)); MFX_TRY(get_event(job, ev + 1, &b));
        spans.push_back(Span{ ev, ev + 1, cls });
        ev += 2;
        CUDA_TRY(cudaEventRecord(a, on));
        return MFX_OK;
    };
    auto timed_end = [&](cudaStream_t on) -> int { CUDA_TRY(cudaEventRecord(job.events[spans.back().b], on)); return MFX_OK; };
    // Two streams (fast precision, light-sampling integrators): the shadow queries of bounce b touch sh_* and rad only,
    // the closest hits of bounce b+1 the ray queue and hit[] only -- side by side, the head of one persistent grid fills
    // the SMs the tail of the other one leaves idle.  shade(b+1) rewrites sh_*: it waits for shadow(b).
    // Measured (C2 / C3, two shadow queues deep): +2.7 % / +4.2 % on frames of 16 M paths (what one of eight GPUs renders),
    // +0.4 % / +1.0 % on the full 133 M-path frame -- so it is used where launches are short and their tails weigh, and big frames keep one
    // stream (and per-kernel event times that do not overlap).  MFX_TWO_STREAMS = 0 / 1 forces either.
    const long two_env = env_long("MFX_TWO_STREAMS", -1);
    const bool two = !exact && !sky && !ctr && (two_env >= 0 ? two_env != 0 : (size_t)tm.n_pix * (size_t)p->spp <= ((size_t)48 << 20));
    if (two && !s->stream2) MFX_TRY(stream_get(s->device, &s->stream2));
    cudaStream_t st2 = two ? s->stream2 : st;
    LaunchCfg cfg2 = cfg; cfg2.stream = st2;
    // ... and with a second shadow queue shade(b+1) does not wait for shadow(b) either: the shadow launches trail the
    // extend / shade chain on their own stream, two queues deep (shade(b) waits for shadow(b-2), which used its queue)
    if (two && s->sh2_P != s->wf.P) {
        CUDA_TRY(cudaStreamSynchronize(st));
        for (int k = 0; k < 3; k++) { dev_free_one(s, s->sh2[k]); s->sh2[k] = nullptr; }
        for (int k = 0; k < 3; k++) MFX_TRY(dev_alloc_t(s, &s->sh2[k], (size_t)s->wf.P));
        s->sh2_P = s->wf.P;
    }
    WaveF wf_alt = s->wf;
    if (two) { wf_alt.sh_o = s->sh2[0]; wf_alt.sh_d = s->sh2[1]; wf_alt.sh_c = s->sh2[2]; }
    // ... and spill columns of their own: a thread's stack column is picked by its block and lane, so a shadow grid and a
    // closest-hit grid beside it would push and pop each other's deferred subtrees (missed occluders, wrong hits)
    const SceneF *sfp_sh = sfp;
    SceneF sf_sh;
    if (two && sfp->stack_spill) {
        if (!s->spill2) MFX_TRY(dev_alloc_t(s, &s->spill2, own_spill_entries(*sfp)));
        sf_sh = *sfp;
        sf_sh.stack_spill = s->spill2;
        sfp_sh = &sf_sh;
    }
    cudaEvent_t e_shadow_done[2] = { nullptr, nullptr };

    const int P = exact ? s->wx.P : s->wf.P;
    const int D = s->max_depth;
    // (own tree, default sampler and uncounted runs only: the instrumented and reference-stream runs keep one launch pair per bounce)
    const int sky_tail = (sky && !exact && !counting && sfp->own_tree && !(p->flags & MFX_SAMPLE_REFERENCE_STREAM)) ? (int)env_long("MFX_SKY_TAIL", 8) : 0;
    const int npix_total = tm.n_pix;
    const int pix_chunk = std::min(npix_total, P);
    const int S_wave = std::max(1, std::min(p->spp, P / std::max(1, pix_chunk)));
    uint32_t launches = 0, l_ext = 0, l_sh = 0;
    int *counts = exact ? s->wx.counts : s->wf.counts;
    for (int pix0 = 0; pix0 < npix_total; pix0 += pix_chunk) {
        const int np = std::min(pix_chunk, npix_total - pix0);
        for (int s0 = 0; s0 < p->spp; s0 += S_wave) {
            const int S = std::min(S_wave, p->spp - s0);
            const int sabs = p->first_sample + s0;
            tm.sshift = 0;                                       // (the exact kernels keep sample-major path ids)
            if (!exact) for (long want = env_long("MFX_SAMPLE_BLOCK_LOG2", 4); tm.sshift < want && S % (2 << tm.sshift) == 0; tm.sshift++) {}
            CUDA_TRY(cudaMemsetAsync(counts, 0, MFX_COUNTS_LEN * sizeof(int), st));
#ifdef MFX_DEBUG_CHECKS
            // (MFX_DEBUG_FAULT=1 leaves the previous call's stamps in place: the next call's shadow rays then look like
            //  second rays of their bounce and the check must trip -- the test that the assertion is alive)
            if (!exact && s->wf.dbg_stamp && !env_long("MFX_DEBUG_FAULT", 0)) CUDA_TRY(cudaMemsetAsync(s->wf.dbg_stamp, 0, (size_t)s->wf.P * sizeof(int), st));
#endif
            cfg.max_items = 0;
            if (exact) mfx_x_raygen(cfg, s->sx, s->wx, tm, pix0, np, sabs, S, p->seed);
            else if (hyb) mfx_h_raygen(cfg, *sfp, s->sx, s->wf, s->wh, tm, pix0, np, sabs, S, p->seed);
            else mfx_f_raygen(cfg, *sfp, s->wf, tm, pix0, np, sabs, S, p->seed);
            launches++;
            for (int b = 0; b <= D; b++) {
                MFX_TRY(timed(0, st));
                if (exact && hyb_x) {
                    const HybQuery q{ sky ? MFX_SKY_TMIN : 1e-6, sky ? MFX_SKY_TMAX : 99999999., sky ? 1 : 0 };
                    mfx_h_extend_x(cfg, s->sf, s->sx, s->sh, s->wx, s->wf, s->wh, b, q);
                    mfx_h_accum_fixups(st, s->wh, job.d_totals + 4);
                    mfx_h_guard(st, s->wf, job.d_totals);
                    launches += 6;
                } else if (exact) mfx_x_extend(cfg, s->sx, s->wx, b, ctr);
                else if (hyb && b == 0) {
                    const HybQuery q{ sky ? MFX_SKY_TMIN : 1e-6, sky ? MFX_SKY_TMAX : 99999999., sky ? 1 : 0 };   // Integrators.fs:108 / RayTracing.fs:368
                    mfx_h_extend(cfg, *sfp, s->sx, s->sh, s->wf, s->wh, 0, q, 0);
                    mfx_h_accum_fixups(st, s->wh, job.d_totals + 4);
                    launches += 2;
                } else mfx_f_extend(cfg, *sfp, s->wf, b, ctr);
                MFX_TRY(timed_end(st));
                if (sky) {      // GetColor (RayTracing.fs:367-382): no light, no shadow query
                    if (exact) mfx_x_shade_sky(cfg, s->sx, s->wx, tm, pix0, np, sabs, b, p->seed);
                    else mfx_f_shade_sky(cfg, *sfp, s->wf, tm, pix0, np, sabs, b, p->seed);
                    launches += 2; l_ext++;
                    // the throughput path hands whatever is still alive after bounce MFX_SKY_TAIL (default 8) to ONE launch
                    // that traces and shades every such path to its end (k_f_trace6<TAIL>): the late bounces hold a few
                    // rays at most and cost launch latency, and the host no longer looks at a queue size inside a Sample
                    if (sky_tail > 0 && b == sky_tail && b < D) {
                        MFX_TRY(timed(0, st));
                        mfx_f_sky_tail(cfg, *sfp, s->wf, tm, pix0, np, sabs, b + 1, p->seed);
                        MFX_TRY(timed_end(st));
                        launches++; l_ext++;
                        break;
                    }
                    // `depth < 50`: the late bounces hold a few rays at most (paths caught inside glass spheres), and a
                    // full persistent grid that finds a tiny queue still costs ~30 us per bounce (profiles/).  A queue
                    // never grows from one bounce to the next, so the host looks at the device-side count now and then
                    // and sizes the following grids for it -- or leaves the loop when nothing is left.
                    if (sky_tail == 0 && b >= 8 && (b % 6) == 2 && b < D) {      // (per-bounce mode only: exact precision, instrumented and reference-stream runs)
                        int next_n = 0;
                        CUDA_TRY(cudaMemcpyAsync(&next_n, counts + b + 1, sizeof(int), cudaMemcpyDeviceToHost, st));
                        CUDA_TRY(cudaStreamSynchronize(st));
                        if (next_n == 0) break;
                        cfg.max_items = next_n;
                    }
                    continue;
                }
                const WaveF &wq = (two && (b & 1)) ? wf_alt : s->wf;           // the shadow queue of this bounce
                if (two && e_shadow_done[b & 1]) CUDA_TRY(cudaStreamWaitEvent(st, e_shadow_done[b & 1], 0));   // shade(b) rewrites the queue shadow(b-2) read
                if (exact) mfx_x_shade(cfg, s->sx, s->wx, tm, pix0, np, sabs, b, p->seed);
                else mfx_f_shade(cfg, *sfp, wq, tm, pix0, np, sabs, b, p->seed);
                if (two) {
                    cudaEvent_t e_shaded;
                    MFX_TRY(get_event(job, ev++, &e_shaded));
                    CUDA_TRY(cudaEventRecord(e_shaded, st));
                    CUDA_TRY(cudaStreamWaitEvent(st2, e_shaded, 0));
                }
                MFX_TRY(timed(1, st2));
                if (exact && hyb_x) mfx_h_shadow_x(cfg, s->sx, s->sf_ref, s->sh, s->wx, b);
                else if (exact) mfx_x_shadow(cfg, s->sx, s->wx, b, ctr);
                else mfx_f_shadow(cfg2, *sfp_sh, wq, b, ctr);
                MFX_TRY(timed_end(st2));
                if (two) {
                    MFX_TRY(get_event(job, ev++, &e_shadow_done[b & 1]));
                    CUDA_TRY(cudaEventRecord(e_shadow_done[b & 1], st2));
                }
                launches += 3; l_ext++; l_sh++;
            }
            for (int k = 0; k < 2; k++)                                          // resolve reads rad: every shadow launch is in
                if (two && e_shadow_done[k]) { CUDA_TRY(cudaStreamWaitEvent(st, e_shadow_done[k], 0)); e_shadow_done[k] = nullptr; }
            if (exact) mfx_x_resolve(cfg, s->sx, s->wx, tm, pix0, np, S, s->d_pixsum);
            else mfx_f_resolve(cfg, *sfp, s->wf, tm, pix0, np, S, s->d_pixsum);
            // rays traced: exact: closest = counts[0..D], shadow = counts[1..D+1];
            //              fast : closest = counts[0..D], shadow = counts[V+2 .. V+2+D]
            if (sky) mfx_accum_ray_totals(st, counts, 0, D + 1, 0, 0, job.d_totals);
            else if (exact) mfx_accum_ray_totals(st, counts, 0, D + 1, 1, D + 1, job.d_totals);
            else mfx_accum_ray_totals(st, counts, 0, D + 1, MFX_MAX_VERTS + 2, D + 1, job.d_totals);
            launches += 2;
        }
    }
    mfx_x_finalize(cfg, s->d_pixsum, s->width, s->height, 0.0, p->spp, tm, d_color_wh, d_rgba);
    launches++;
    CUDA_TRY(cudaEventRecord(e_end, st));
    CUDA_TRY(cudaGetLastError());
    // the statistics follow the kernels down the stream into pinned host memory: nobody has to block for them
    CUDA_TRY(cudaMemcpyAsync(job.h_totals, job.d_totals, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(job.h_ctr, job.d_ctr, sizeof(TravCounters), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaEventRecord(job.done, st));
    if (ordered) {
        std::lock_guard<std::mutex> g(g_order_mu);
        cudaEvent_t &tail = g_frame_tail[s->device];
        if (!tail) CUDA_TRY(cudaEventCreateWithFlags(&tail, cudaEventDisableTiming));
        CUDA_TRY(cudaEventRecord(tail, st));
    }
    job.launches = launches; job.l_ext = l_ext; job.l_sh = l_sh;
    job.active = true; job.has_copy = false;
    if (trace_host) fprintf(stderr, "[mfx] launch_sample dev %d: layouts/buffers ready after %.3f ms, %d launches + %zu events enqueued after %.3f ms\n",
                            s->device, th_prepared, launches, ev, th_ms());
    return MFX_OK;
}

// Waits for a launched Sample call (and its texture download, if it has one) and publishes its MfxStats.
static int finish_sample(MfxScene *s, FrameJob &job)
{
    if (!job.active) return MFX_OK;
    job.active = false;
    const auto tf0 = std::chrono::steady_clock::now();
    CUDA_TRY(cudaEventSynchronize(job.done));
    const auto tf1 = std::chrono::steady_clock::now();
    if (job.has_copy) CUDA_TRY(cudaEventSynchronize(job.copied));
    if (env_long("MFX_DEBUG", 0) >= 2)
        fprintf(stderr, "[mfx] finish_sample dev %d: waited %.3f ms for the kernels, %.3f ms more for the download\n", s->device,
                std::chrono::duration<double, std::milli>(tf1 - tf0).count(), std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tf1).count());
    const unsigned long long *totals = job.h_totals;
    const TravCounters &hc = *job.h_ctr;
    MfxStats &stt = s->stats;
    memset(&stt, 0, sizeof(stt));
    stt.closest_rays = totals[0]; stt.shadow_rays = totals[1]; stt.paths = totals[2];
    if (totals[3]) return fail(MFX_ERR_CUDA, "traversal watchdog tripped in %llu warp(s): the frame is incomplete", totals[3]);
    if (totals[5]) return fail(MFX_ERR_CUDA, "debug build: %llu index / shadow-ray check(s) failed in the wavefront kernels", totals[5]);
    for (int c = 0; c < 2; c++) { stt.nodes[c] = hc.v[c][0]; stt.tris[c] = hc.v[c][1]; stt.spheres[c] = hc.v[c][2]; }
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, job.events[job.e_begin], job.events[job.e_end]));
    stt.ms_total = ms;
    double m_ext = 0., m_sh = 0.;
    for (const Span &sp : job.spans) {
        CUDA_TRY(cudaEventElapsedTime(&ms, job.events[sp.a], job.events[sp.b]));
        if (sp.cls == 0) m_ext += ms; else m_sh += ms;
    }
    stt.ms_extend = m_ext; stt.ms_shadow = m_sh; stt.ms_shade = stt.ms_total - m_ext - m_sh;
    stt.launches = job.launches; stt.launches_extend = job.l_ext; stt.launches_shadow = job.l_sh;
    stt.hybrid_fixups = (uint32_t)std::min<unsigned long long>(totals[4], 0xffffffffull);
    return MFX_OK;
}

static int finish_oldest(MfxScene *s)
{
    if (s->job_count == 0) return MFX_OK;
    FrameJob &j = s->jobs[s->job_head];
    s->job_head = (s->job_head + 1) % 2;
    s->job_count--;
    return finish_sample(s, j);
}

// The synchronous call: one Sample, finished before it returns.  Frames still in flight from the async entry point are
// completed first (their textures fill, their statistics are superseded).
static int run_sample(MfxScene *s, const MfxSampleParams *p, double *d_color_wh, float4 *d_rgba)
{
    if (!s || !p) return fail(MFX_ERR_INVALID_ARGUMENT, "null scene/params");
    while (s->job_count > 0) MFX_TRY(finish_oldest(s));
    MFX_TRY(launch_sample(s, p, d_color_wh, d_rgba, s->jobs[0]));
    return finish_sample(s, s->jobs[0]);
}

static int ensure_pinned(MfxScene *, size_t bytes)
{
    if (g_pinned_bytes >= bytes) return MFX_OK;
    if (g_pinned) { cudaFreeHost(g_pinned); g_pinned = nullptr; g_pinned_bytes = 0; }
    CUDA_TRY(cudaMallocHost(&g_pinned, bytes));
    g_pinned_bytes = bytes;
    return MFX_OK;
}

// D2H into a caller buffer: direct when the caller registered it (mfx_host_register), else
// through the scene's pinned staging buffer.
static int copy_out(MfxScene *s, void *host, const void *dev, size_t bytes)
{
    cudaPointerAttributes attr;
    bool pinned = (cudaPointerGetAttributes(&attr, host) == cudaSuccess) && (attr.type == cudaMemoryTypeHost);
    cudaGetLastError();
    if (pinned) {
        CUDA_TRY(cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, s->stream));
        CUDA_TRY(cudaStreamSynchronize(s->stream));
    } else {
        std::lock_guard<std::mutex> g(g_pool_mu);
        MFX_TRY(ensure_pinned(s, bytes));
        CUDA_TRY(cudaMemcpyAsync(g_pinned, dev, bytes, cudaMemcpyDeviceToHost, s->stream));
        CUDA_TRY(cudaStreamSynchronize(s->stream));
        memcpy(host, g_pinned, bytes);
    }
    return MFX_OK;
}

extern "C" int mfx_pixel_integrator_sample(MfxScene *s, const MfxSampleParams *p, double *texture)
{
    if (!texture) return fail(MFX_ERR_INVALID_ARGUMENT, "null texture");
    if (!s) return fail(MFX_ERR_INVALID_ARGUMENT, "null scene");
    MFX_TRY(bind_device(s->device)); MFX_TRY(ensure_frame_buffers(s));
    MFX_TRY(run_sample(s, p, s->d_color_wh, nullptr));
    return copy_out(s, texture, s->d_color_wh, (size_t)s->width * s->height * 4 * sizeof(double));
}

extern "C" int mfx_pixel_integrator_sample_device(MfxScene *s, const MfxSampleParams *p, void *d_rgba_f32)
{
    if (!d_rgba_f32) return fail(MFX_ERR_INVALID_ARGUMENT, "null device buffer");
    if (!s) return fail(MFX_ERR_INVALID_ARGUMENT, "null scene");
    return run_sample(s, p, nullptr, (float4 *)d_rgba_f32);
}

// IPixelIntegrator.Sample without the wait: the kernels and the download of Color[w,h] are enqueued and the call returns.
// Up to two frames may be in flight per scene -- the download of frame k (copy stream, its own device buffer) then runs
// beside the kernels of frame k+1; a third call first completes the oldest frame.
extern "C" int mfx_pixel_integrator_sample_async(MfxScene *s, const MfxSampleParams *p, double *texture)
{
    if (!texture) return fail(MFX_ERR_INVALID_ARGUMENT, "null texture");
    if (!s) return fail(MFX_ERR_INVALID_ARGUMENT, "null scene");
    MFX_TRY(bind_device(s->device));
    cudaPointerAttributes attr;
    const bool pinned = (cudaPointerGetAttributes(&attr, texture) == cudaSuccess) && (attr.type == cudaMemoryTypeHost);
    cudaGetLastError();
    if (!pinned) return fail(MFX_ERR_INVALID_ARGUMENT, "mfx_pixel_integrator_sample_async needs a pinned texture: register it once with mfx_host_register");
    MFX_TRY(ensure_frame_buffers(s));
    if (s->job_count == 2) MFX_TRY(finish_oldest(s));
    const int slot = (s->job_head + s->job_count) % 2;
    const size_t bytes = (size_t)s->width * s->height * 4 * sizeof(double);
    if (!s->d_color_async[slot]) MFX_TRY(dev_alloc(s, (void **)&s->d_color_async[slot], bytes));
    if (!s->copy_stream) MFX_TRY(stream_get(s->device, &s->copy_stream));
    FrameJob &job = s->jobs[slot];
    MFX_TRY(launch_sample(s, p, s->d_color_async[slot], nullptr, job));
    CUDA_TRY(cudaStreamWaitEvent(s->copy_stream, job.done, 0));
    CUDA_TRY(cudaMemcpyAsync(texture, s->d_color_async[slot], bytes, cudaMemcpyDeviceToHost, s->copy_stream));
    CUDA_TRY(cudaEventRecord(job.copied, s->copy_stream));
    job.has_copy = true;
    s->job_count++;
    return MFX_OK;
}

// Completes the OLDEST frame in flight: its texture is filled and mfx_get_stats describes it.  No frame in flight: no-op.
extern "C" int mfx_pixel_integrator_wait(MfxScene *s)
{
    if (!s) return fail(MFX_ERR_INVALID_ARGUMENT, "null scene");
    MFX_TRY(bind_device(s->device));
    return finish_oldest(s);
}

extern "C" int mfx_pixel_integrator_sample_device_color(MfxScene *s, const MfxSampleParams *p, void *d_color_wh_f64)
{
    if (!d_color_wh_f64) return fail(MFX_ERR_INVALID_ARGUMENT, "null device buffer");
    if (!s) return fail(MFX_ERR_INVALID_ARGUMENT, "null scene");
    return run_sample(s, p, (double *)d_color_wh_f64, nullptr);
}

extern "C" int mfx_pixel_integrator_sample_f32(MfxScene *s, const MfxSampleParams *p, float *rgba)
{
    if (!rgba) return fail(MFX_ERR_INVALID_ARGUMENT, "null output");
    if (!s) return fail(MFX_ERR_INVALID_ARGUMENT, "null scene");
    MFX_TRY(bind_device(s->device)); MFX_TRY(ensure_frame_buffers(s));
    MFX_TRY(run_sample(s, p, nullptr, s->d_rgba));
    return copy_out(s, rgba, s->d_rgba, (size_t)s->width * s->height * sizeof(float4));
}

extern "C" int mfx_get_stats(const MfxScene *s, MfxStats *out)
{
    if (!s || !out) return fail(MFX_ERR_INVALID_ARGUMENT, "null argument");
    *out = s->stats;
    return MFX_OK;
}

extern "C" int mfx_host_register(void *ptr, uint64_t bytes)
{
    if (!ptr || !bytes) return fail(MFX_ERR_INVALID_ARGUMENT, "null buffer");
    MFX_TRY(ensure_device());
    CUDA_TRY(cudaHostRegister(ptr, bytes, cudaHostRegisterPortable));     // pinned for every device: mfx_multi_sample DMAs from all of them
    return MFX_OK;
}
extern "C" int mfx_host_unregister(void *ptr)
{
    if (!ptr) return fail(MFX_ERR_INVALID_ARGUMENT, "null buffer");
    MFX_TRY(ensure_device());
    CUDA_TRY(cudaHostUnregister(ptr));
    return MFX_OK;
}

// ------------------------------------------------------------------ finer seams
template <typename F>
static int with_ray_buffers(MfxScene *s, int64_t n, const double *a, size_t a_per, const double *b, size_t b_per,
                            int32_t *prim, int32_t *sub, double *t, F launch)
{
    double *da = nullptr, *db = nullptr, *dt = nullptr; int *dp = nullptr, *ds = nullptr;
    int rc = MFX_OK;
    auto cleanup = [&]() { cudaFree(da); cudaFree(db); cudaFree(dt); cudaFree(dp); cudaFree(ds); };
#define WRB_TRY(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { cleanup(); return fail(MFX_ERR_CUDA, "%s failed: %s", #x, cudaGetErrorString(e_)); } } while (0)
    // every copy rides on the scene's stream (created non-blocking: the legacy default stream orders nothing against it)
    if (a) { WRB_TRY(cudaMalloc(&da, n * a_per * sizeof(double))); WRB_TRY(cudaMemcpyAsync(da, a, n * a_per * sizeof(double), cudaMemcpyHostToDevice, s->stream)); }
    if (b) { WRB_TRY(cudaMalloc(&db, n * b_per * sizeof(double))); WRB_TRY(cudaMemcpyAsync(db, b, n * b_per * sizeof(double), cudaMemcpyHostToDevice, s->stream)); }
    WRB_TRY(cudaMalloc(&dt, n * sizeof(double))); WRB_TRY(cudaMalloc(&dp, n * sizeof(int)));
    if (sub) WRB_TRY(cudaMalloc(&ds, n * sizeof(int)));
    launch(da, db, dp, ds, dt);
    WRB_TRY(cudaGetLastError());
    WRB_TRY(cudaMemcpyAsync(prim, dp, n * sizeof(int), cudaMemcpyDeviceToHost, s->stream));
    WRB_TRY(cudaMemcpyAsync(t, dt, n * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    if (sub) WRB_TRY(cudaMemcpyAsync(sub, ds, n * sizeof(int), cudaMemcpyDeviceToHost, s->stream));
    WRB_TRY(cudaStreamSynchronize(s->stream));
#undef WRB_TRY
    cleanup();
    return rc;
}

// The fast-precision seams run the PRODUCTION wavefront traversal kernel: the rays go through the wave's
// queues in chunks of its capacity (bounce 0, closest or shadow queue), exactly like rays of a frame.  src (device, per
// ray, nullptr: none): the slot id of the primitive the ray starts on, or -1.
static void fast_seam(MfxScene *s, const SceneF *sfp, const LaunchCfg &cfg, int any_hit, int64_t n, const double *o, const double *d, const double *uv,
                      const int *src, float tmin, float tmax, int *prim, int *sub, double *t)
{
    WaveF w = s->wf;
    w.tmin = tmin;
    w.tmax = tmax;
    w.cam_origin = 0;
    for (int64_t first = 0; first < n; first += w.P) {
        const int m = (int)std::min<int64_t>(w.P, n - first);
        cudaMemsetAsync(w.counts, 0, MFX_COUNTS_LEN * sizeof(int), s->stream);
        mfx_f_seam_setup(cfg, *sfp, w, m, o, d, uv, src, first, tmax, any_hit);
        if (any_hit) mfx_f_shadow(cfg, *sfp, w, 0, nullptr); else mfx_f_extend(cfg, *sfp, w, 0, nullptr);
        mfx_f_seam_read(cfg, *sfp, w, m, first, any_hit, prim, sub, t);
    }
}

// The same seams through the id-exact hybrid kernel (closest-hit queries only): f64 rays into the wave's ray64 queue.
static void hybrid_seam(MfxScene *s, const SceneF *sfp, const LaunchCfg &cfg, int64_t n, const double *o, const double *d, const double *uv,
                        double tmin, double tmax, int *prim, int *sub, double *t)
{
    WaveF w = s->wf;
    w.cam_origin = 0;
    const HybQuery q{ tmin, tmax, s->integrator == MFX_SKY_TRACER ? 1 : 0 };
    for (int64_t first = 0; first < n; first += w.P) {
        const int m = (int)std::min<int64_t>(w.P, n - first);
        cudaMemsetAsync(w.counts, 0, MFX_COUNTS_LEN * sizeof(int), s->stream);
        mfx_h_seam_setup(cfg, s->sx, w, s->wh, m, o, d, uv, first);
        mfx_h_extend(cfg, *sfp, s->sx, s->sh, w, s->wh, 0, q, 1);
        mfx_h_seam_read(cfg, s->sx, s->wh, m, first, prim, sub, t);
        int fx = 0;     // seam calls are synchronous anyway: keep the number of rays the exact walk had to settle
        if (cudaMemcpyAsync(&fx, s->wh.fix_n, sizeof(int), cudaMemcpyDeviceToHost, s->stream) == cudaSuccess && cudaStreamSynchronize(s->stream) == cudaSuccess)
            s->stats.hybrid_fixups = (first == 0 ? 0u : s->stats.hybrid_fixups) + (uint32_t)fx;
    }
}

extern "C" int mfx_bvh_hit(MfxScene *s, int32_t precision, int32_t any_hit, int64_t n, const double *origins, const double *dirs,
                           double tmin, double tmax, int32_t *prim, int32_t *sub, double *t)
{
    if (!s || !origins || !dirs || !prim || !t) return fail(MFX_ERR_INVALID_ARGUMENT, "mfx_bvh_hit: null argument");
    if (n <= 0) return MFX_OK;
    MFX_TRY(bind_device(s->device));
    LaunchCfg cfg{ s->sm_count, 128, s->stream, 0, 0 };
    if (precision == MFX_EXACT_F64) {
        MFX_TRY(flatten_exact(s));
        return with_ray_buffers(s, n, origins, 3, dirs, 3, prim, sub, t, [&](double *o, double *d, int *p, int *sb, double *tt) {
            mfx_x_bvh_hit(cfg, s->sx, any_hit, n, o, d, tmin, tmax, p, sb, tt);
        });
    } else if (precision == MFX_FAST_F32) {
        MFX_TRY(flatten_fast(s));
        const SceneF *sfp = &s->sf;
        MFX_TRY(ensure_wave_fast(s, (size_t)n));
        const bool hyb = !any_hit && use_hybrid(0);
        if (hyb) { MFX_TRY(flatten_hybrid(s)); MFX_TRY(ensure_wave_hybrid(s)); }
        return with_ray_buffers(s, n, origins, 3, dirs, 3, prim, sub, t, [&](double *o, double *d, int *p, int *sb, double *tt) {
            if (hyb) hybrid_seam(s, sfp, cfg, n, o, d, nullptr, tmin, tmax, p, sb, tt);
            else fast_seam(s, sfp, cfg, any_hit, n, o, d, nullptr, nullptr, (float)tmin, (float)tmax, p, sb, tt);
        });
    }
    return fail(MFX_ERR_INVALID_ARGUMENT, "unknown precision %d", precision);
}

// Rays that start on a surface, as the rays of bounces >= 1 and the shadow rays of a fast frame: always k_f_trace6 (the
// id-exact kernel only ever traces bounce 0, whose rays have no source).
extern "C" int mfx_bvh_hit_from(MfxScene *s, int32_t any_hit, int64_t n, const double *origins, const double *dirs, const int32_t *src,
                                double tmin, double tmax, int32_t *prim, int32_t *sub, double *t)
{
    if (!s || !origins || !dirs || !prim || !t) return fail(MFX_ERR_INVALID_ARGUMENT, "mfx_bvh_hit_from: null argument");
    if (n <= 0) return MFX_OK;
    const int np = (int)s->prims.size();
    if (src)
        for (int64_t r = 0; r < n; r++)
            if (src[r] < -1 || src[r] >= np) return fail(MFX_ERR_INVALID_ARGUMENT, "mfx_bvh_hit_from: src[%lld] = %d outside [-1, %d)", (long long)r, src[r], np);
    MFX_TRY(bind_device(s->device));
    LaunchCfg cfg{ s->sm_count, 128, s->stream, 0, 0 };
    MFX_TRY(flatten_fast(s));
    MFX_TRY(ensure_wave_fast(s, (size_t)n));
    int *dsrc = nullptr;
    if (src) {
        // the id leaf_f3 compares with a ray's src is b.w of the primitive's slots without the half bit, and the own
        // tree's slots carry the caller's index there (build_own_tree_host: make_fast_slots(prims[i], i, ..)), so the
        // caller's indices go to the device as they are
        cudaError_t e = cudaMalloc(&dsrc, (size_t)n * sizeof(int));
        if (e == cudaSuccess) e = cudaMemcpyAsync(dsrc, src, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, s->stream);
        if (e != cudaSuccess) { cudaFree(dsrc); return fail(MFX_ERR_CUDA, "mfx_bvh_hit_from: source ids: %s", cudaGetErrorString(e)); }
    }
    const int rc = with_ray_buffers(s, n, origins, 3, dirs, 3, prim, sub, t, [&](double *o, double *d, int *p, int *sb, double *tt) {
        fast_seam(s, &s->sf, cfg, any_hit, n, o, d, nullptr, dsrc, (float)tmin, (float)tmax, p, sb, tt);
    });
    cudaFree(dsrc);
    return rc;
}

extern "C" int mfx_trace_primary(MfxScene *s, int32_t precision, int64_t n, const double *uv, int32_t *prim, double *t)
{
    if (!s || !prim || !t) return fail(MFX_ERR_INVALID_ARGUMENT, "mfx_trace_primary: null argument");
    if (!uv && n != (int64_t)s->width * s->height) return fail(MFX_ERR_INVALID_ARGUMENT, "uv == NULL needs n == width*height");
    if (n <= 0) return MFX_OK;
    MFX_TRY(bind_device(s->device));
    LaunchCfg cfg{ s->sm_count, 128, s->stream, 0, 0 };
    if (precision == MFX_EXACT_F64) {
        MFX_TRY(flatten_exact(s));
        return with_ray_buffers(s, n, uv, 2, nullptr, 0, prim, nullptr, t, [&](double *u, double *, int *p, int *, double *tt) {
            mfx_x_primary(cfg, s->sx, n, u, p, tt);
        });
    } else if (precision == MFX_FAST_F32) {
        MFX_TRY(flatten_fast(s));
        const SceneF *sfp = &s->sf;
        MFX_TRY(ensure_wave_fast(s, (size_t)n));
        const bool hyb = use_hybrid(0);
        if (hyb) { MFX_TRY(flatten_hybrid(s)); MFX_TRY(ensure_wave_hybrid(s)); }
        return with_ray_buffers(s, n, uv, 2, nullptr, 0, prim, nullptr, t, [&](double *u, double *, int *p, int *, double *tt) {
            const bool sky = (s->integrator == MFX_SKY_TRACER);      // ListHit(ray, 0.00001, 10000000), RayTracing.fs:368
            if (hyb) { hybrid_seam(s, sfp, cfg, n, nullptr, nullptr, u, sky ? MFX_SKY_TMIN : 1e-6, sky ? MFX_SKY_TMAX : 99999999., p, nullptr, tt); return; }
            fast_seam(s, sfp, cfg, 0, n, nullptr, nullptr, u, nullptr, sky ? (float)MFX_SKY_TMIN : 1e-6f, sky ? (float)MFX_SKY_TMAX : 99999999.f, p, nullptr, tt);
        });
    }
    return fail(MFX_ERR_INVALID_ARGUMENT, "unknown precision %d", precision);
}

// ------------------------------------------------------------------ Film (Film.fs:13-34)
// One device's film.  The steps below touch the pixels `tm` owns: the whole frame for mfx_film_*, a device's column
// stripes for mfx_multi_film_*.  The buffers are not in the scene's buffer pool (dev_alloc): an mfx_multi_sample_async may
// be growing a replica's pool list on its worker thread while the caller destroys a film.
struct FilmBuffers {
    double *d_sum = nullptr, *d_target = nullptr;   // Color[w,h], x-major
    uint8_t *d_rgba8 = nullptr;                     // row-major
};

struct MfxFilm {
    MfxScene *scene;
    FilmBuffers buf;
    double frame_count = 0.;
};

static void film_free(MfxScene *s, FilmBuffers &b)
{
    cudaSetDevice(s->device);
    cudaFree(b.d_sum); cudaFree(b.d_target); cudaFree(b.d_rgba8);
    b = FilmBuffers();
}

static int film_alloc(MfxScene *s, FilmBuffers &b)
{
    MFX_TRY(bind_device(s->device));
    const size_t npx = (size_t)s->width * s->height;
    auto alloc3 = [&]() {
        return cudaMalloc(&b.d_sum, 4 * npx * sizeof(double)) == cudaSuccess && cudaMalloc(&b.d_target, 4 * npx * sizeof(double)) == cudaSuccess &&
               cudaMalloc(&b.d_rgba8, 4 * npx) == cudaSuccess;
    };
    if (alloc3()) return MFX_OK;
    cudaGetLastError();     // memory parked in the buffer pool is not in use: give it back and retry once
    film_free(s, b);
    pool_trim(s->device);
    if (alloc3()) return MFX_OK;
    cudaGetLastError();
    film_free(s, b);
    return fail(MFX_ERR_OUT_OF_MEMORY, "film allocation failed");
}

static int film_reset(MfxScene *s, const FilmBuffers &b)
{
    const size_t bytes = (size_t)s->width * s->height * 4 * sizeof(double);
    CUDA_TRY(cudaMemsetAsync(b.d_sum, 0, bytes, s->stream));
    CUDA_TRY(cudaMemsetAsync(b.d_target, 0, bytes, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return MFX_OK;
}

// Film.GetFrame (Film.fs:18-23): one Sample into the scene's Color[w,h], then sum += frame, target = sum / frame_count
static int film_frame(MfxScene *s, const TileMap &tm, const FilmBuffers &b, const MfxSampleParams *p, double frame_count)
{
    MFX_TRY(ensure_frame_buffers(s));
    MFX_TRY(run_sample(s, p, s->d_color_wh, nullptr));
    mfx_film_add(s->stream, tm, s->width, b.d_sum, s->d_color_wh, b.d_target, frame_count);
    CUDA_TRY(cudaGetLastError());
    return MFX_OK;
}

// ACES (Scene.fs:315-330), or under MFX_SKY_TRACER the sphere sample's sqrt(c) flipped vertically (RayTracing.fs:456-460)
static int film_screen(MfxScene *s, const TileMap &tm, const FilmBuffers &b)
{
    if (s->integrator == MFX_SKY_TRACER) mfx_film_display_sky(s->stream, tm, s->width, b.d_target, b.d_rgba8);
    else mfx_film_tonemap(s->stream, tm, s->width, b.d_target, b.d_rgba8);
    CUDA_TRY(cudaGetLastError());
    return MFX_OK;
}

// target = sum / frameCount (Film.fs:23) after an import: Film.AddSample of a zero frame with the restored count
static int film_retarget(MfxScene *s, const TileMap &tm, const FilmBuffers &b, double frame_count)
{
    if (frame_count > 0.) {
        MFX_TRY(ensure_frame_buffers(s));
        CUDA_TRY(cudaMemsetAsync(s->d_color_wh, 0, (size_t)s->width * s->height * 4 * sizeof(double), s->stream));
        mfx_film_add(s->stream, tm, s->width, b.d_sum, s->d_color_wh, b.d_target, frame_count);
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaStreamSynchronize(s->stream));
    }
    return MFX_OK;
}

extern "C" int mfx_film_create(MfxScene *s, MfxFilm **out)
{
    if (!s || !out) return fail(MFX_ERR_INVALID_ARGUMENT, "null argument");
    FilmBuffers b;
    MFX_TRY(film_alloc(s, b));
    *out = new MfxFilm{ s, b };
    return mfx_film_reset(*out);
}

extern "C" int mfx_film_destroy(MfxFilm *f)
{
    if (!f) return MFX_OK;
    cudaSetDevice(f->scene->device);
    cudaStreamSynchronize(f->scene->stream);
    film_free(f->scene, f->buf);
    delete f;
    return MFX_OK;
}

extern "C" int mfx_film_reset(MfxFilm *f)                      // Film.Reset, Film.fs:26-30
{
    if (!f) return fail(MFX_ERR_INVALID_ARGUMENT, "null film");
    MFX_TRY(bind_device(f->scene->device));
    f->frame_count = 0.;
    return film_reset(f->scene, f->buf);
}

extern "C" int mfx_film_get_frame(MfxFilm *f, const MfxSampleParams *p, double *texture)   // Film.fs:18-23,32-34
{
    if (!f || !p) return fail(MFX_ERR_INVALID_ARGUMENT, "null argument");
    MfxScene *s = f->scene;
    MFX_TRY(bind_device(s->device));
    MFX_TRY(film_frame(s, stripe_tilemap(s->width, s->height, 0, 0, 1), f->buf, p, f->frame_count + 1.));
    f->frame_count += 1.;
    if (texture) return copy_out(s, texture, f->buf.d_target, (size_t)s->width * s->height * 4 * sizeof(double));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return MFX_OK;
}

extern "C" int mfx_film_post_process(MfxFilm *f, uint8_t *rgba8)   // Scene.fs:315-330
{
    if (!f || !rgba8) return fail(MFX_ERR_INVALID_ARGUMENT, "null argument");
    MfxScene *s = f->scene;
    MFX_TRY(bind_device(s->device));
    MFX_TRY(film_screen(s, stripe_tilemap(s->width, s->height, 0, 0, 1), f->buf));
    return copy_out(s, rgba8, f->buf.d_rgba8, (size_t)s->width * s->height * 4);
}

extern "C" int mfx_film_frame_count(const MfxFilm *f, double *out)
{
    if (!f || !out) return fail(MFX_ERR_INVALID_ARGUMENT, "null argument");
    *out = f->frame_count;
    return MFX_OK;
}

extern "C" int mfx_film_export(MfxFilm *f, double *sum, double *frame_count)
{
    if (!f || !sum || !frame_count) return fail(MFX_ERR_INVALID_ARGUMENT, "null argument");
    MFX_TRY(bind_device(f->scene->device));
    *frame_count = f->frame_count;
    return copy_out(f->scene, sum, f->buf.d_sum, (size_t)f->scene->width * f->scene->height * 4 * sizeof(double));
}

extern "C" int mfx_film_import(MfxFilm *f, const double *sum, double frame_count)
{
    if (!f || !sum || frame_count < 0.) return fail(MFX_ERR_INVALID_ARGUMENT, "bad argument");
    MfxScene *s = f->scene;
    MFX_TRY(bind_device(s->device));
    CUDA_TRY(cudaMemcpyAsync(f->buf.d_sum, sum, (size_t)s->width * s->height * 4 * sizeof(double), cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    f->frame_count = frame_count;
    return film_retarget(s, stripe_tilemap(s->width, s->height, 0, 0, 1), f->buf, frame_count);
}

#include "mfx_multi.inl"
