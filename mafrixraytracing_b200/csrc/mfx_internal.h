// mfx_internal.h -- structures shared by the host orchestration (mfx_host.cpp) and the two
// kernel translation units (mfx_exact.cu: f64, --fmad=false; mfx_fast.cu: f32).
// Nothing here crosses the C ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define MFX_LEAF_NODE_COUNT 3      // Bvh.LeafNodeCount, BvhNode.fs:39
#define MFX_REJECTION_CAP 128      // cap of the GetRandomInUnitSphere loop (Material.fs:12), see DESIGN.md
#define MFX_MAX_VERTS 64           // max_depth + 1 shaded vertices per path (max_depth <= 63; the sphere sample uses 50)
#define MFX_MODE_SKY 2             // MFX_SKY_TRACER: GetColor of RenderTest/Sample/RayTracing.fs:367-382
#define MFX_SKY_TMIN 0.00001       // ListHit(hitable, ray, 0.00001, 10000000), RayTracing.fs:368
#define MFX_SKY_TMAX 10000000.
#define MFX_STACK_SMEM_MAX 48      // own-tree stack entries in shared memory: [48][128 threads] x 8 B = the 48 KB a block
                                   // gets without opting in to more (MFX_STACK_SMEM is capped there)

// ------------------------------------------------------------------ exact (f64) device layout
// One BvhNode, heap-indexed like the reference (children 2i+1 / 2i+2).  64 B.
struct __align__(16) NodeX {
    double pmin[3];
    double pmax[3];
    int    first;
    int    count;
    double pad;
};
// One IHitable in LEAF ORDER (the reference's `indices` indirection is applied at flatten time,
// ref_id[] maps a slot back to the original primitive).  e1=v1-v0, e2=v2-v0, e3=v3-v0 are the
// same single subtractions Triangle.PreCalcu performs per call (Trangle.fs:124-125), so storing
// them is bit-neutral.  Sphere: v0 = center, e1[0] = radius.  112 B.
struct __align__(16) PrimX {
    double v0[3];
    double e1[3];
    double e2[3];
    double e3[3];
    int    kind;
    int    material;
    double pad;
};
struct MatX {
    int    kind;
    int    pad;
    double albedo[3];
    double fuzz, ei, et;
};
struct TriSampleX { double v0[3], e1[3], e2[3]; };
struct LightX {
    TriSampleX t1, t2;      // Rect(p0,p1,p2,p3) = Triangle(p0,p1,p2) + Triangle(p0,p2,p3)
    double area;            // rect.area = t1.area + t2.area
    double normal[3];
    double color[3];
};
struct CamX { double pos[3], topleft[3], right[3], down[3]; };
// MFX_SKY_TRACER: RayTraceCamera (RayTracing.fs:335-364) rides in CamX as pos = origin, topleft = lowerLeftCorner,
// right = horizontal, down = vertical -- GetRay's `lowerLeftCorner + s*horizontal + t*vertical - origin` has the
// shape of the pinhole's `topleft + u*right + v*down - pos` -- plus the lens basis and radius.
struct LensX { double u[3], v[3], radius; };

struct SceneX {
    const NodeX *nodes;
    const PrimX *prims;
    const int   *ref_id;
    const MatX  *mats;
    LightX light;
    CamX   cam;
    LensX  lens;                    // MFX_SKY_TRACER
    const double *perlin_rf;        // MFX_SKY_TRACER: Perlin.ranfloat[256] (RayTracing.fs:82) or null
    const int    *perlin_perm;      //                 perm_x | perm_y | perm_z [3*256] (:83-85) or null
    int    width, height, max_depth, mode;
    int    n_prims;
};

// Per-wave path state, exact mode (SoA over P paths).
struct WaveX {
    int     P;              // capacity
    double *ray_o;          // [3][P]
    double *ray_d;          // [3][P]
    double *hit_t;          // [P]
    int    *hit_slot;       // [P]  slot | sub<<30, or -1
    double *sh_d;           // [3][P] unit direction to the light sample
    double *sh_dist;        // [P]
    double *v_l;            // [V][3][P]  l_k   (direct term, zeroed by the shadow kernel when occluded);
                            //            MFX_SKY_TRACER: [3][P] the colour the recursion bottoms out with
    double *v_col;          // [V][3][P]  col_k
    double *v_ei;           // [V][P]     Lambertian.Shade cosine (mode B)
    int    *v_kind;         // [V][P]     material kind at vertex k (mode B)
    int    *nv;             // [P] number of shaded vertices
    int    *queue[2];       // ping-pong queues of path ids
    int    *counts;         // [MFX_MAX_VERTS+2] queue sizes per bounce
};

// ------------------------------------------------------------------ fast (f32) device layout
// Children pair of interior heap node i: 64 B = 4 x float4.
//   q0 = (L.min.x, L.min.y, L.min.z, L.max.x)   q1 = (L.max.y, L.max.z, R.min.x, R.min.y)
//   q2 = (R.min.z, R.max.x, R.max.y, R.max.z)   q3 = (metaL, metaR, -, -) as int bits
// meta >= 0: leaf,  first<<3 | count (count <= 6 fast slots);  meta < 0: interior.
// Boxes are rounded outward from the f64 bounds.
struct __align__(16) PairF { float4 q0, q1, q2, q3; };
// One 128 B record per node of the library's OWN tree (SceneF.own_tree = 1): the boxes of its (up to) four children,
// SoA so one lane tests four boxes from four 32 B loads.  The tree is a binned-SAH BVH over the fast slots collapsed to
// four children per node.  The tree only decides the visiting order -- a nearest-hit query has one
// answer whichever BVH finds it -- so MFX_FAST_F32 is free to use a better one than the reference's median split
// (BvhNode.fs:42-61), which MFX_EXACT_F64 keeps because its tie rules are tree-shaped (quirk Q1).  Meta:
//   meta >= 0: leaf (first<<3 | count), MFX_QUAD_EMPTY: empty slot, other negatives: interior, child record = ~meta.
struct __align__(16) QuadF { float4 lox, hix, loy, hiy, loz, hiz, meta, pad; };
#define MFX_QUAD_EMPTY ((int)0x80000000)
// One fast primitive slot, 48 B = 3 x float4, leaf order.
//   triangle: a = (v0.xyz, kind bits), b = (e1.xyz, -), c = (e2.xyz, -)
//   sphere  : a = (center.xyz, kind 2), b = (radius, r^2, -, prim)
//   big sphere (r >= 32): a = (radius as f64 bit pair, -, kind 3), b = (cx f64 pair, -, prim), c = (cy pair, cz pair)
struct __align__(16) SlotF { float4 a, b, c; };
struct MatF { float albedo[3]; int kind; float fuzz, ei, et, pad; };
struct LightF {
    float v0a[3], e1a[3], e2a[3];
    float v0b[3], e1b[3], e2b[3];
    float area, inv_pdf;    // inv_pdf = area (pdf_li = 1/area)
    float normal[3];
    float color[3];
};
struct CamF { float pos[3], topleft[3], right[3], down[3]; };

struct SceneF {
    const PairF *pairs;     // indexed by the interior node's 1-based heap index h (siblings share a 128 B line)
    const QuadF *quads;     // own tree only: its records (see QuadF)
    const SlotF *slots;     // leaf order (rects split in two)
    const int   *slot_prim; // slot -> leaf-order primitive (exact slot) ; sub in bit 30
    const int   *ref_id;    // exact slot -> original primitive index
    const float4 *slot_nrm; // geometric normal per fast slot (xyz), w = material as int bits
    const MatF  *mats;
    LightF light;
    CamF   cam;
    CamX   camx;            // f64 camera: primary rays are generated in f64 and rounded once
    LensX  lens;            // MFX_SKY_TRACER (see SceneX)
    const float *perlin_rf; // MFX_SKY_TRACER: noise tables (f32 view) or null
    const int   *perlin_perm;
    float  root_min[3], root_max[3];
    int    root_meta;       // leaf meta if the whole tree is one leaf, else -1
    int    width, height, max_depth, mode;
    int    n_slots;
    int    n_quads, n_mats;     // record / material counts (bounds of the debug build's checks)
    int    levels;          // entries of the per-level entry-distance column (deepest child depth + 1)
    int    has_big_sphere;  // any kind-3 slot (selects the kernel variant with the f64 sphere branch)
    int    own_tree;        // 0: pairs follow the reference tree (heap-indexed); 1: quads are the SAH 4-wide tree
    int    own_depth;       // own tree: number of quad levels (deferred-hit stack holds <= 3 per level)
    int    stack_smem;      // own tree: stack entries kept in shared memory per thread (<= MFX_STACK_SMEM_MAX)
    uint2 *stack_spill;     // own tree: [3*own_depth - stack_smem][spill_threads] overflow entries (null if none); every
                            // launch that may run beside another one needs columns of its own
    int    spill_threads;
};

// Path state lives at QUEUE POSITIONS, not at path ids: the shade kernel of bounce b reads entry i of buffer b&1 and
// writes the survivors densely into buffer (b+1)&1 (and the shadow rays densely into sh_*), so every kernel of the
// next bounce reads consecutive entries -- no queue of path ids, no gather.  The path id (pixel/sample for the RNG,
// slot of `rad`) rides in ray_d.w / sh_c.w.
struct WaveF {
    int     P;
    float4 *ray_o[2];       // [P] o.xyz, w = source fast slot as int bits (-1: camera)
    float4 *ray_d[2];       // [P] d.xyz, w = path id as int bits
    float4 *thr[2];         // [P] throughput rgb (not stored for bounce 0: it is 1)
    float2 *hit;            // [P] (t, slot as int bits) of the extend-queue entry
    float4 *rad;            // [P] accumulated radiance rgb, indexed by PATH ID
    float4 *sh_o;           // [P] shadow ray origin.xyz, w = source fast slot
    float4 *sh_d;           // [P] shadow dir.xyz, w = dist
    float4 *sh_c;           // [P] contribution rgb if unoccluded, w = path id as int bits
    float   tmin;           // tMin of every query (1e-6, Integrators.fs:44,108; the Bvh.Hit seam may pass another)
    float   tmax;           // tMax of the closest-hit queries (99999999., Integrators.fs:108; 1e7 for the sky tracer)
    int     cam_origin;     // 1: every bounce-0 ray starts at the camera position (pinhole): ray_o is neither written by
                            //    raygen nor read by the bounce-0 extend / shade (own-tree frames only; 0 for the seams)
    int    *dbg_stamp;      // MFX_DEBUG_CHECKS: [P] last bounce that queued a shadow ray for the path (null otherwise)
    int    *counts;         // [0 .. MFX_MAX_VERTS+1] extend queue sizes per bounce,
                            // [MFX_MAX_VERTS+2 + bounce] shadow queue sizes
};
// + [2(V+2)+b] extend queue cursors, [3(V+2)+b] shadow queue cursors (persistent kernels);
// the last entry is the traversal watchdog flag
#define MFX_COUNTS_LEN (4 * (MFX_MAX_VERTS + 2))
// one before the watchdog flag: violations counted by a `make DEBUG=1` build (MFX_DEBUG_CHECKS: bounds of every index the
// wavefront kernels compute, one shadow ray per path and bounce) -- compute-sanitizer is closed on the GPU pool
#define MFX_DBG_SLOT (MFX_COUNTS_LEN - 2)

// ------------------------------------------------------------------ hybrid (id-exact closest hit, mfx_hybrid.cu)
// The closest-hit query of the reference has ONE answer (BvhNode.fs:62-83): the smallest t over every primitive the
// exhaustive walk tests, ties to the later leaf in depth-first order, then to the earlier slot of that leaf.  The
// hybrid kernel finds it on the library's own SAH tree: f32 slab tests over boxes padded per ray (conservative
// against every rounding between the f64 ray and the f32 arithmetic), candidate primitives tested with the exact
// kernel's f64 functions on the exact layout's PrimX records, the tie rule applied from the reference tree's leaf
// table, and the winner's reference leaf box re-tested with AABB.hit verbatim (the reference only ever tests a
// primitive whose boxes all pass; child boxes nest, so the leaf's own test decides).  Anything that check does not
// clear goes to the exact kernel's traversal (k_h_fixup).
// One own-tree slot in f64: the PrimX arithmetic inputs (v0, e1 = v1-v0, e2 = v2-v0, e3 = v3-v0: the single subtractions
// Triangle.PreCalcu does per call, Trangle.fs:124-125) in the own tree's slot order, so a leaf's records are adjacent.
//   kind 0: Triangle, or first triangle of a Rect;  kind 1: second triangle of a Rect (e1, e2, e3 all present: Rect.Hit
//   tries (v0,e1,e2) first, Rect.fs:26-31);  kind 2: Sphere (v0 = center, e1[0] = radius).  ref = exact leaf-order slot.
struct __align__(16) PrimH {
    double v0[3];
    double e1[3];
    double e2[3];
    double e3[3];
    int    kind;
    int    ref;
    double pad;
};
struct SceneH {
    const PrimH *prims_h;       // [own-tree fast slots]
    const int  *leaf_of_ref;    // exact slot -> heap index of the reference-tree leaf holding it (BvhNode.fs:40-41)
    const int2 *ref_fslot;      // exact slot -> own-tree fast slots of (first, second) triangle; .y = -1 unless a Rect
    float max_abs;              // largest |coordinate| of the scene bound: scale of the per-ray box pad
    int   n_ref;                // number of exact slots (= primitives)
    float pad_factor;           // 4e-6 (MFX_HYB_PAD_PPB = 4000 parts per billion): the margin experiment of tools/hyb_pad_margin.py
};
#define MFX_HYB_FIX_CAP (1 << 20)
struct WaveH {
    double *dir64;              // [P][3] f64 direction of the queued closest-hit rays (bounce 0 / the seams)
    double *org64;              // [P][3] f64 origin; not touched by pinhole frames (WaveF.cam_origin: the camera position)
    double *t;                  // [P] exact hit distance
    int    *ref;                // [P] exact slot | sub << 30, -1 = miss, -2 = waiting for k_h_fixup
    int    *fix_q;              // [MFX_HYB_FIX_CAP] queue positions waiting for k_h_fixup
    int    *fix_n;              // [1] how many were flagged (may exceed the capacity: then k_h_fixup scans `ref`)
};

// Traversal counters (instrumented runs only): [class][nodes,tris,spheres]
struct TravCounters { unsigned long long v[2][3]; };

// Which pixels this rank renders, and in which order (local index pl -> pixel):
//   pix != null : table of linear pixel ids (interleaved square tiles, mfx_tile_map);
//   stripe > 0  : COLUMN STRIPES computed arithmetically -- stripe c (columns [c*stripe, (c+1)*stripe)) belongs to rank
//                 c % world; local order = owned stripe after owned stripe, row-major inside a stripe.  In the reference's
//                 x-major Color[w,h] (Texture.fs:21-28) a stripe is one contiguous block, so a GPU's share of the frame
//                 goes to the host with one strided copy and nothing has to be uploaded or reduced (mfx_multi_sample);
//   otherwise   : identity (the whole frame).
struct TileMap {
    const int *pix;
    int  n_pix;
    int  stripe, rank, world, height;
    int  sshift;            // fast wavefront: path ids keep 2^sshift samples of one pixel next to each other (path_split)
};

// ------------------------------------------------------------------ launchers (defined in the .cu TUs)
// max_items > 0: the host knows an upper bound of the queue this launch works on (sky tracer, late bounces): the
// persistent grid is clamped to the blocks that many entries can occupy
struct LaunchCfg { int blocks; int threads; cudaStream_t stream; int reference_stream; int max_items; };

// exact
void mfx_x_raygen(const LaunchCfg &, const SceneX &, const WaveX &, TileMap tm, int pix0, int npix, int s0, int S,
                  uint64_t seed);
void mfx_x_extend(const LaunchCfg &, const SceneX &, const WaveX &, int bounce, TravCounters *ctr);
void mfx_x_shade(const LaunchCfg &, const SceneX &, const WaveX &, TileMap tm, int pix0, int npix, int s0,
                 int bounce, uint64_t seed);
void mfx_x_shadow(const LaunchCfg &, const SceneX &, const WaveX &, int bounce, TravCounters *ctr);
void mfx_x_resolve(const LaunchCfg &, const SceneX &, const WaveX &, TileMap tm, int pix0, int npix, int S,
                   double *pixsum /* [w*h][4] row-major */);
void mfx_x_bvh_hit(const LaunchCfg &, const SceneX &, int any_hit, long long n, const double *o, const double *d,
                   double tmin, double tmax, int *prim, int *sub, double *t);
void mfx_x_primary(const LaunchCfg &, const SceneX &, long long n, const double *uv, int *prim, double *t);
void mfx_x_shade_sky(const LaunchCfg &, const SceneX &, const WaveX &, TileMap tm, int pix0, int npix, int s0,
                     int bounce, uint64_t seed);
void mfx_x_finalize(const LaunchCfg &, const double *pixsum, int width, int height, double inv_unused, int spp,
                    TileMap tm, double *color_wh /* x-major Color[w,h] or null */, float4 *rgba_f32 /* row-major or null */);

// fast
void mfx_f_raygen(const LaunchCfg &, const SceneF &, const WaveF &, TileMap tm, int pix0, int npix, int s0, int S,
                  uint64_t seed);
void mfx_f_extend(const LaunchCfg &, const SceneF &, const WaveF &, int bounce, TravCounters *ctr);
void mfx_f_sky_tail(const LaunchCfg &, const SceneF &, const WaveF &, TileMap tm, int pix0, int npix, int s0, int bounce, uint64_t seed);
void mfx_f_shade(const LaunchCfg &, const SceneF &, const WaveF &, TileMap tm, int pix0, int npix, int s0,
                 int bounce, uint64_t seed);
void mfx_f_shadow(const LaunchCfg &, const SceneF &, const WaveF &, int bounce, TravCounters *ctr);
void mfx_f_shade_sky(const LaunchCfg &, const SceneF &, const WaveF &, TileMap tm, int pix0, int npix, int s0,
                     int bounce, uint64_t seed);
void mfx_f_resolve(const LaunchCfg &, const SceneF &, const WaveF &, TileMap tm, int pix0, int npix, int S,
                   double *pixsum);
void mfx_f_seam_setup(const LaunchCfg &, const SceneF &, const WaveF &, int n, const double *o, const double *d, const double *uv,
                      const int *src, long long first, float tmax, int any_hit);
void mfx_f_seam_read(const LaunchCfg &, const SceneF &, const WaveF &, int n, long long first, int any_hit, int *prim, int *sub, double *t);

// hybrid (mfx_hybrid.cu, --fmad=false): id-exact closest hits on the own tree
struct HybQuery { double tmin, tmax; int sky; };
void mfx_h_raygen(const LaunchCfg &, const SceneF &, const SceneX &, const WaveF &, const WaveH &, TileMap tm, int pix0, int npix,
                  int s0, int S, uint64_t seed);
void mfx_h_seam_setup(const LaunchCfg &, const SceneX &, const WaveF &, const WaveH &, int n, const double *o, const double *d,
                      const double *uv, long long first);
void mfx_h_extend(const LaunchCfg &, const SceneF &, const SceneX &, const SceneH &, const WaveF &, const WaveH &, int bounce, HybQuery q, int seam);
void mfx_h_seam_read(const LaunchCfg &, const SceneX &, const WaveH &, int n, long long first, int *prim, int *sub, double *t);
void mfx_h_accum_fixups(cudaStream_t, const WaveH &, unsigned long long *total);
// the closest-hit queries of an MFX_EXACT_F64 wave (queue `bounce` of WaveX) through the hybrid kernel
void mfx_h_guard(cudaStream_t, const WaveF &, unsigned long long *totals);
// the shadow queries of an MFX_EXACT_F64 wave: f32 walk of the reference tree's copy, exact decision at every visited leaf
void mfx_h_shadow_x(const LaunchCfg &, const SceneX &, const SceneF &ref_layout, const SceneH &, const WaveX &, int bounce);
void mfx_h_extend_x(const LaunchCfg &, const SceneF &, const SceneX &, const SceneH &, const WaveX &, const WaveF &, const WaveH &, int bounce, HybQuery q);

// misc (mfx_fast.cu)
// totals[0] += sum counts[ext_lo..+ext_n), totals[1] += sum counts[sh_lo..+sh_n), totals[2] += counts[0]
void mfx_accum_ray_totals(cudaStream_t, const int *counts, int ext_lo, int ext_n, int sh_lo, int sh_n,
                          unsigned long long *totals);
// Film kernels over the pixels tm owns (column stripes; one stripe of the frame's width = the whole frame)
void mfx_film_add(cudaStream_t, TileMap tm, int width, double *sum, const double *frame, double *target, double frame_count);
void mfx_film_tonemap(cudaStream_t, TileMap tm, int width, const double *target_wh, uint8_t *rgba8);
void mfx_film_display_sky(cudaStream_t, TileMap tm, int width, const double *target_wh, uint8_t *rgba8);
