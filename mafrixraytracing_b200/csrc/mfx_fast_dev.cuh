// mfx_fast_dev.cuh -- f32 device helpers shared by the wavefront kernels (mfx_fast.cu) and the id-exact hybrid
// traversal (mfx_hybrid.cu): ray setup, 256-bit record loads, queue-count indices, and the own tree's child order,
// traversal stack and launch geometry.
#pragma once
#include "mfx_device.cuh"
#include <algorithm>

typedef V3<float> F3;

#define FAST_BLOCK 128
#define FAST_LEVELS 30

__device__ __forceinline__ F3 f3(float x, float y, float z) { return mk3<float>(x, y, z); }
__device__ __forceinline__ float4 ldg4(const float4 *p) { return __ldg(p); }
// One 256-bit read-only load (sm_100: LDG.E.256): two adjacent float4 of a 32-byte aligned pair.  A divergent warp
// pays the L1 per 32-byte sector touched, so fetching a record as 4 x 32 B instead of 7 x 16 B halves that cost.
__device__ __forceinline__ void ldg8(const float4 *p, float4 &a, float4 &b)
{
    asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "l"(p));
}

struct RayF {
    F3 o, d, idir, ood;
    float tmin;
    int src;    // leaf-order primitive the ray starts on (never re-hit a planar source), -1 none
};

__device__ __forceinline__ float safe_rcp(float d)
{
    const float eps = 1e-30f;
    return 1.0f / (fabsf(d) > eps ? d : copysignf(eps, d));
}

__device__ __forceinline__ RayF make_ray(F3 o, F3 d, float tmin, int src)
{
    RayF r; r.o = o; r.d = d; r.tmin = tmin; r.src = src;
    r.idir = f3(safe_rcp(d.x), safe_rcp(d.y), safe_rcp(d.z));
    r.ood = f3(o.x * r.idir.x, o.y * r.idir.y, o.z * r.idir.z);
    return r;
}

// slab test; returns entry distance, hit iff entry <= exit
__device__ __forceinline__ bool box_f(const RayF &r, float lx, float ly, float lz, float hx, float hy, float hz,
                                      float tmax, float &entry)
{
    const float x0 = fmaf(lx, r.idir.x, -r.ood.x), x1 = fmaf(hx, r.idir.x, -r.ood.x);
    const float y0 = fmaf(ly, r.idir.y, -r.ood.y), y1 = fmaf(hy, r.idir.y, -r.ood.y);
    const float z0 = fmaf(lz, r.idir.z, -r.ood.z), z1 = fmaf(hz, r.idir.z, -r.ood.z);
    const float tn = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fmaxf(fminf(z0, z1), r.tmin));
    const float tf = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fminf(fmaxf(z0, z1), tmax));
    entry = tn;
    return tn <= tf;
}

// Intersects the slots of one leaf: Moller-Trumbore with the reference's acceptance rules
// (Trangle.fs:130-148) folded into one predicate (no early exits: every lane of a leaf vote runs the
// same instructions), the stable quadratic of Sphere.fs:21-43 for spheres.
__device__ __forceinline__ float rcp_approx(float x)
{
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ RayF make_ray_fast(F3 o, F3 d, float tmin, int src)
{
    RayF r; r.o = o; r.d = d; r.tmin = tmin; r.src = src;
    const float eps = 1e-30f;
    r.idir = f3(rcp_approx(fabsf(d.x) > eps ? d.x : copysignf(eps, d.x)),
                rcp_approx(fabsf(d.y) > eps ? d.y : copysignf(eps, d.y)),
                rcp_approx(fabsf(d.z) > eps ? d.z : copysignf(eps, d.z)));
    r.ood = f3(o.x * r.idir.x, o.y * r.idir.y, o.z * r.idir.z);
    return r;
}


#define CNT_SH(b)  (MFX_MAX_VERTS + 2 + (b))
#define CUR_EXT(b) (2 * (MFX_MAX_VERTS + 2) + (b))
#define CUR_SH(b)  (3 * (MFX_MAX_VERTS + 2) + (b))

#define KEY_INF 0x7f800000u

__device__ __forceinline__ unsigned umin_(unsigned a, unsigned b) { return a < b ? a : b; }
__device__ __forceinline__ unsigned umax_(unsigned a, unsigned b) { return a > b ? a : b; }
__device__ __forceinline__ int pick4(const float4 &m, unsigned id)
{
    const float lo = (id & 1u) ? m.y : m.x, hi = (id & 1u) ? m.w : m.z;
    return __float_as_int((id & 2u) ? hi : lo);
}

// ---------------------------------------------------------------- persistent warps (k_f_trace4, k_f_trace6, k_h_trace)
// Watchdog: the loop is bounded so a logic error can never hang the GPU; a trip raises the flag in counts[] (Sample fails).
__device__ __forceinline__ bool watchdog_tripped(unsigned &iters, unsigned limit, int *counts)
{
    if (++iters <= limit) return false;
    if ((threadIdx.x & 31u) == 0) atomicAdd(&counts[MFX_COUNTS_LEN - 1], 1);
    return true;
}

// Ray replacement: once >= T lanes of the warp are idle (and the queue is not exhausted) the warp claims that many of the n
// queue entries with one atomicAdd on the cursor (ballot / popc / shuffle); an idle lane whose entry exists takes it as
// `pid` (the ray lives at its queue position) and runs start().  `exhausted` is set once a claim reaches the end of the
// queue.  Returns the mask of the lanes still idle.  A batch of refills pays one cursor round trip for many rays, and rays
// that start together are neighbours in the queue.
template <typename Start>
__device__ __forceinline__ unsigned warp_refill(unsigned idle, int T, int *cursor, int n, bool &exhausted, int &pid, Start start)
{
    if (exhausted || __popc(idle) < T) return idle;
    const unsigned lane = threadIdx.x & 31u;
    const int nidle = __popc(idle);
    int base = 0;
    if (lane == 0) base = atomicAdd(cursor, nidle);
    base = __shfl_sync(0xffffffffu, base, 0);
    if (base + nidle >= n) exhausted = true;
    if (pid < 0) {
        const int idx = base + __popc(idle & ((1u << lane) - 1u));
        if (idx < n) { pid = idx; start(); }
    }
    return __ballot_sync(0xffffffffu, pid < 0);
}

// Leaf vote: the lanes in `leaves` run their leaf tests
// once >= T of them hold a leaf, or no lane has node work left.
__device__ __forceinline__ bool leaf_vote(unsigned leaves, unsigned idle, int T)
{
    return leaves && (__popc(leaves) >= T || (~idle & ~leaves) == 0u);
}

// ---------------------------------------------------------------- the own tree's traversal stack (k_f_trace6, k_h_trace)
// Child order of a node step: the sorting network (0,1)(2,3)(0,2)(1,3)(1,2) over the four slot keys, k0 nearest.
__device__ __forceinline__ void sort4(const unsigned (&key)[4], unsigned &k0, unsigned &k1, unsigned &k2, unsigned &k3)
{
    const unsigned a0 = umin_(key[0], key[1]), a1 = umax_(key[0], key[1]);
    const unsigned a2 = umin_(key[2], key[3]), a3 = umax_(key[2], key[3]);
    k0 = umin_(a0, a2); const unsigned t2 = umax_(a0, a2);
    const unsigned t1 = umin_(a1, a3); k3 = umax_(a1, a3);
    k1 = umin_(t1, t2); k2 = umax_(t1, t2);
}

// One thread's stack of deferred hits.  An entry is (sort key of the child, record that holds it); the key's low bits are
// leaf << 2 | slot.  Entries [0, S) sit in dynamic shared memory as [entry][thread] (conflict free: my_stack = s_stack +
// threadIdx.x), deeper ones in the thread's global spill column (my_spill = stack_spill + blockIdx.x * FAST_BLOCK +
// threadIdx.x, stride spill_threads: own_tree_blocks keeps a launch inside the columns own_spill_entries sized).
__device__ __forceinline__ void own_put(uint2 *my_stack, uint2 *my_spill, int S, size_t spill_stride, int i, uint2 v,
                                        const SceneF &sc, int *counts)
{
    DBG_CHECK(i >= 0 && i < 3 * sc.own_depth, counts);
    DBG_CHECK(i < S || blockIdx.x * FAST_BLOCK + threadIdx.x < (unsigned)sc.spill_threads, counts);
    if (i < S) my_stack[(size_t)i * FAST_BLOCK] = v; else my_spill[(size_t)(i - S) * spill_stride] = v;
}

// Defers the hits behind the one a node step consumes now (k1..k3 sorted, KEY_INF: none) with record `node`, nearest on top.
__device__ __forceinline__ int own_push(uint2 *my_stack, uint2 *my_spill, int S, size_t spill_stride, int sp,
                                        unsigned k1, unsigned k2, unsigned k3, int node, const SceneF &sc, int *counts)
{
    const int m = (k1 != KEY_INF ? 1 : 0) + (k2 != KEY_INF ? 1 : 0) + (k3 != KEY_INF ? 1 : 0);
    if (m >= 1) own_put(my_stack, my_spill, S, spill_stride, sp + m - 1, make_uint2(k1, (unsigned)node), sc, counts);
    if (m >= 2) own_put(my_stack, my_spill, S, spill_stride, sp + m - 2, make_uint2(k2, (unsigned)node), sc, counts);
    if (m >= 3) own_put(my_stack, my_spill, S, spill_stride, sp, make_uint2(k3, (unsigned)node), sc, counts);
    return sp + m;
}

// Pops the deepest entry whose entry distance is <= limit (ANY: the top one, never culls) and re-reads its child link from
// the record that holds it.
struct OwnPop {
    int sp;         // stack height after the pop
    int link;       // the child's link: leaf meta, or ~record of an interior child
    bool found;     // false: the stack ran empty
    bool leaf;
};
template <bool ANY>
__device__ __forceinline__ OwnPop own_pop(const uint2 *my_stack, const uint2 *my_spill, int S, size_t spill_stride, int sp,
                                          float limit, const SceneF &sc, int *counts)
{
    OwnPop r;
    for (;;) {
        if (sp == 0) { r.sp = 0; r.found = false; r.leaf = false; r.link = 0; return r; }
        --sp;
        const uint2 e = (sp < S) ? my_stack[(size_t)sp * FAST_BLOCK] : my_spill[(size_t)(sp - S) * spill_stride];
        if (ANY || __uint_as_float(e.x & ~7u) <= limit) {
            const int link = __ldg(reinterpret_cast<const int *>(&sc.quads[e.y].meta) + (e.x & 3u));
            DBG_CHECK(e.y < (unsigned)sc.n_quads && ((e.x & 4u) ? (link >= 0 && (link >> 3) + (link & 7) <= sc.n_slots) : (unsigned)~link < (unsigned)sc.n_quads), counts);
            r.sp = sp; r.link = link; r.found = true; r.leaf = (e.x & 4u) != 0;
            return r;
        }
    }
}

// Launch geometry of the own-tree kernels: the shared part of the stack as dynamic shared memory, a persistent grid that
// never runs more threads than the spill columns were sized for, nor more blocks than max_items entries can occupy.
static_assert(MFX_STACK_SMEM_MAX * FAST_BLOCK * sizeof(uint2) <= 48 * 1024, "the own-tree stack must launch without a shared-memory opt-in");
static inline size_t own_stack_smem(const SceneF &sc) { return (size_t)sc.stack_smem * FAST_BLOCK * sizeof(uint2); }
template <typename K>
static inline int own_tree_blocks(K kernel, const LaunchCfg &c, const SceneF &sc)
{
    int blocks = persistent_blocks(kernel, FAST_BLOCK, c.blocks, own_stack_smem(sc));
    if (sc.stack_spill && blocks * FAST_BLOCK > sc.spill_threads) blocks = sc.spill_threads / FAST_BLOCK;
    if (c.max_items > 0) blocks = std::max(1, std::min(blocks, (c.max_items + FAST_BLOCK - 1) / FAST_BLOCK));
    return blocks;
}
