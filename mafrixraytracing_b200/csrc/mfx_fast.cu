// mfx_fast.cu -- MFX_FAST_F32 wavefront kernels (the throughput path) + small utility kernels.
//
// Layouts (mfx_internal.h, built by mfx_host.cpp / mfx_build.cpp):
//   * own tree (default): 128 B records of four child boxes + links over a binned-SAH BVH of the fast slots,
//     48 B primitive slots in that tree's leaf order, 16 B normal+material side array for the shade kernel;
//   * reference tree (instrumented counting runs): 64 B children pairs indexed by the reference's heap index
//     (BvhNode.fs:40-41), slots in its leaf order.
// Traversal kernels: one ray per lane in persistent warps, ordered descent, t-shrink, ray replacement from the
// bounce's queue, vote-postponed leaf tests.
//   k_f_trace6  own tree, sorted 4-wide node step, stack of (key, record) entries in shared memory   <- shipped
//   k_f_trace4  reference tree, binary, stackless (1 bit per level): the COUNT-instrumented kernel
// Path state lives at QUEUE POSITIONS (WaveF, mfx_internal.h): entry i of buffer b & 1 is the i-th ray of bounce b, the
// shade kernel writes its survivors densely into the other buffer and its shadow rays densely into sh_*; no queue of
// path ids, no gathers.
// Shading: k_f_shade (BSDF + light sample, block-aggregated position claims), k_f_shade_sky (the sphere sample's
// GetColor, MFX_SKY_TRACER); k_f_raygen / k_f_resolve bracket a wave.
#include "mfx_device.cuh"
#include <algorithm>

#include "mfx_fast_dev.cuh"

// Big sphere (r >= 32, e.g. the r = 1000 ground sphere of the RayTracing.fs scenes): |o - c| ~ r makes
// the f32 quadratic lose ~1e-4 of t, so this one primitive kind is solved in f64 (Sphere.fs:21-43
// verbatim: b = 2 oc.d, c = oc.oc - r^2, q = -0.5 (b -+ sqrt(b^2 - 4c))).  Kept out of line so its f64
// registers do not cost the traversal loop its occupancy.
__device__ __noinline__ bool big_sphere_roots(const SlotF *sp, F3 o, F3 d, float &lo, float &hi, float &hb)
{
    const float4 a = ldg4(&sp->a), b = ldg4(&sp->b), c4 = ldg4(&sp->c);
    const double cx = __hiloint2double(__float_as_int(b.y), __float_as_int(b.x));
    const double cy = __hiloint2double(__float_as_int(c4.y), __float_as_int(c4.x));
    const double cz = __hiloint2double(__float_as_int(c4.w), __float_as_int(c4.z));
    const double rad = __hiloint2double(__float_as_int(a.y), __float_as_int(a.x));
    const double ox = (double)o.x - cx, oy = (double)o.y - cy, oz = (double)o.z - cz;
    const double h2 = ox * (double)d.x + oy * (double)d.y + oz * (double)d.z;
    const double cc = ox * ox + oy * oy + oz * oz - rad * rad;
    const double disc = h2 * h2 - cc;
    const double root = sqrt(fmax(disc, 0.0));
    const double q = (h2 < 0.0) ? -(h2 - root) : -(h2 + root);
    const double t1 = (q != 0.0) ? cc / q : q;
    lo = (float)fmin(q, t1); hi = (float)fmax(q, t1); hb = (float)h2;
    return disc > 0.0;
}

template <bool COUNT, bool BIG>
__device__ __forceinline__ bool leaf_f3(const SceneF &sc, const RayF &r, int meta, float &best_t, int &best_slot,
                                        unsigned long long *ctr)
{
    const int first = meta >> 3, cnt = meta & 7;
    bool any = false;
    for (int k = 0; k < cnt; k++) {
        const SlotF *sp = sc.slots + first + k;
        const float4 a = ldg4(&sp->a);
        const float4 b = ldg4(&sp->b);
        const int prim = __float_as_int(b.w) & 0x3fffffff;
        if (__float_as_int(a.w) < 2) {
            const float4 c = ldg4(&sp->c);
            if (COUNT) ctr[1]++;
            const F3 e1 = f3(b.x, b.y, b.z), e2 = f3(c.x, c.y, c.z);
            const F3 s1 = cross(r.d, e2);
            const float div = dot(s1, e1);
            const float inv = rcp_approx(div);
            const F3 dd = r.o - f3(a.x, a.y, a.z);
            const float b1 = dot(dd, s1) * inv;
            const F3 s2 = cross(dd, e1);
            const float b2 = dot(r.d, s2) * inv;
            const float t = dot(e2, s2) * inv;
            // Trangle.fs:130-148 acceptance rules, evaluated without early exits
            const bool ok = (fabsf(div) >= 1e-6f) & (b1 >= 0.f) & (b1 <= 1.f) & (b2 >= 0.f) & ((b1 + b2) < 1.f) &
                            (t > r.tmin) & (t < best_t) & (prim != r.src);
            if (ok) { best_t = t; best_slot = first + k; any = true; }
        } else {
            if (COUNT) ctr[2]++;
            float lo, hi, hb;
            bool real;
            if (BIG && __float_as_int(a.w) == 3) {
                real = big_sphere_roots(sp, r.o, r.d, lo, hi, hb);
            } else {
                const F3 oc = r.o - f3(a.x, a.y, a.z);
                hb = dot(oc, r.d);
                const F3 perp = oc - r.d * hb;              // residual form of the discriminant (robust in f32)
                const float disc = b.y - dot(perp, perp);
                real = disc > 0.f;
                const float root = sqrtf(fmaxf(disc, 0.f));
                const float q = (hb < 0.f) ? -(hb - root) : -(hb + root);
                const float cc = dot(oc, oc) - b.y;
                const float t1 = (q != 0.f) ? cc / q : q;
                lo = fminf(q, t1); hi = fmaxf(q, t1);
            }
            // a ray leaving a convex surface outward cannot re-hit it; one entering takes the far root.  Near grazing the
            // f32 discriminant of a ray that starts on the sphere (hb^2, against rounding of r^2) can come out <= 0:
            // the entering ray then takes the chord -2 hb, which an origin on the surface gives exactly
            const bool src = (prim == r.src);
            if (src && !real && hb < 0.f) { real = true; hi = -2.f * hb; }
            if (real) {
                bool skip = false;
                if (src) { skip = (hb >= 0.f); lo = -1.f; }
                float t = -1.f;
                if (lo >= r.tmin && lo < best_t) t = lo;
                else if (hi > r.tmin && hi < best_t) t = hi;
                if (!skip && t > 0.f) { best_t = t; best_slot = first + k; any = true; }
            }
        }
    }
    return any;
}

// ---------------------------------------------------------------- kernels
__device__ __forceinline__ F3 normalize_f(F3 a)
{
    const float l2 = len2(a);
    const float inv = (l2 > 0.f) ? rsqrtf(l2) : 0.f;
    return a * inv;
}

__device__ __forceinline__ F3 camera_dir_f64(const CamX &c, double u, double v)
{
    // generated in f64 with the reference's operation order (Camera.fs:134-139), rounded once
    const double tx = (c.topleft[0] + c.right[0] * u) + c.down[0] * v - c.pos[0];
    const double ty = (c.topleft[1] + c.right[1] * u) + c.down[1] * v - c.pos[1];
    const double tz = (c.topleft[2] + c.right[2] * u) + c.down[2] * v - c.pos[2];
    const double l = sqrt(tx * tx + ty * ty + tz * tz);
    return f3((float)(tx / l), (float)(ty / l), (float)(tz / l));
}

__global__ void __launch_bounds__(256) k_f_raygen(SceneF sc, WaveF w, TileMap tm, int pix0, int npix, int s0, int S, uint64_t seed)
{
    const long long total = (long long)npix * S;
    for (long long pid = (long long)blockIdx.x * blockDim.x + threadIdx.x; pid < total; pid += (long long)gridDim.x * blockDim.x) {
        int sl, pl;
        path_split(tm, pid, npix, sl, pl);
        int pix, px, py;
        pixel_of(tm, sc.width, pix0 + pl, pix, px, py);
        uint32_t o4[4];
        philox4x32_10((uint32_t)pix, (uint32_t)(s0 + sl), MFX_DIM_CAMERA, 0, (uint32_t)seed, (uint32_t)(seed >> 32), o4);
        const double u = ((double)px + u32_to_unit_f64(o4[0])) / (double)sc.width;
        const double v = ((double)py + u32_to_unit_f64(o4[1])) / (double)sc.height;
        F3 d;
        if (sc.mode == MFX_MODE_SKY && sc.lens.radius != 0.0) {
            // RayTraceCamera.GetRay with a lens sample (RayTracing.fs:360-364), f64, rounded once.  RandomInUnitDisk
            // (:327-333) on the exact mode's stream: (dim 0, iter 1, 2, ..)
            double dx = 0., dy = 0.;
            for (uint32_t it = 0; it < MFX_REJECTION_CAP; it++) {
                uint32_t l4[4];
                philox4x32_10((uint32_t)pix, (uint32_t)(s0 + sl), MFX_DIM_CAMERA, 1u + it, (uint32_t)seed, (uint32_t)(seed >> 32), l4);
                const double a = 2.0 * u32_to_unit_f64(l4[0]) - 1.0, b = 2.0 * u32_to_unit_f64(l4[1]) - 1.0;
                if (a * a + b * b < 1.0) { dx = a; dy = b; break; }
            }
            dx *= sc.lens.radius; dy *= sc.lens.radius;
            const double ox = sc.lens.u[0] * dx + sc.lens.v[0] * dy, oy = sc.lens.u[1] * dx + sc.lens.v[1] * dy, oz = sc.lens.u[2] * dx + sc.lens.v[2] * dy;
            const CamX &c = sc.camx;
            const double tx = (c.topleft[0] + c.right[0] * u) + c.down[0] * v - c.pos[0] - ox;
            const double ty = (c.topleft[1] + c.right[1] * u) + c.down[1] * v - c.pos[1] - oy;
            const double tz = (c.topleft[2] + c.right[2] * u) + c.down[2] * v - c.pos[2] - oz;
            const double l = sqrt(tx * tx + ty * ty + tz * tz);
            d = f3((float)(tx / l), (float)(ty / l), (float)(tz / l));
            w.ray_o[0][pid] = make_float4((float)(c.pos[0] + ox), (float)(c.pos[1] + oy), (float)(c.pos[2] + oz), __int_as_float(-1));
        } else {
            d = camera_dir_f64(sc.camx, u, v);
            if (!w.cam_origin) w.ray_o[0][pid] = make_float4(sc.cam.pos[0], sc.cam.pos[1], sc.cam.pos[2], __int_as_float(-1));
        }
        w.ray_d[0][pid] = make_float4(d.x, d.y, d.z, __int_as_float((int)pid));     // bounce 0: queue position == path id
        // throughput starts at 1: vertex 0 of k_f_shade knows that and the 16 B per path are neither written nor read
        w.rad[pid] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (pid == 0) w.counts[0] = (int)total;
    }
}


// ---------------------------------------------------------------- persistent-warp traversal
// The first kernel (one ray per thread, grid-stride) kept only 5-8 of 32 lanes busy on secondary
// bounces (profiles/r01_v1_baseline_summary.md).  This one keeps every warp resident and
//   (1) REPLACES finished rays: when >= TRACE4_REFILL_T lanes are idle the warp claims that many queue
//       entries with one atomicAdd (ballot/popc/shuffle) and the idle lanes start new rays;
//   (2) POSTPONES leaf tests by vote: a lane that reached leaves parks them (two leaf metas in
//       registers) and idles until >= TRACE4_LEAF_T lanes hold leaves or nobody has node work left, so
//       the (branch-free) triangle tests run with many lanes instead of one or two;
//   (3) keeps the node step branch-light: the descend decision is a handful of selects, the push
//       of the far child is a predicated shared store, the level is tracked in a register; only
//       the pop of deferred siblings is a short divergent loop, run after the leaf vote so it
//       sees the freshly shrunk best_t.
// Per-lane traversal state: heap index, 32-bit trail, level, best hit -- all registers; the far
// child's entry distance per level sits in shared memory ([level][thread], conflict free).
// A watchdog bounds the loop so a logic error can never hang the GPU (flag in counts[]).
// The kernel runs the instrumented counting runs only: it always counts (records fetched, triangle and sphere tests).
constexpr int TRACE4_REFILL_T = 12, TRACE4_LEAF_T = 16, TRACE4_NSTEP = 2;
template <bool ANY, bool BIG>
__global__ void __launch_bounds__(FAST_BLOCK) k_f_trace4(SceneF sc, WaveF w, int bounce, TravCounters *ctr)
{
    extern __shared__ float s_dyn[];
    float *lvl_entry = s_dyn + threadIdx.x;
    const unsigned FULL = 0xffffffffu;
    const int n = ANY ? w.counts[CNT_SH(bounce)] : w.counts[bounce];
    const float4 *ro = ANY ? w.sh_o : w.ray_o[bounce & 1], *rd = ANY ? w.sh_d : w.ray_d[bounce & 1];
    int *cursor = &w.counts[ANY ? CUR_SH(bounce) : CUR_EXT(bounce)];
    unsigned long long local[3] = { 0, 0, 0 };

    int pid = -1;
    RayF r;
    float best_t = 0.f; int best_slot = -1;
    unsigned h = 1u, pend = 0u, depth = 0u;
    bool needPop = false;
    int leafA = -1, leafB = -1; float eB = 0.f;
    bool exhausted = false;
    unsigned iters = 0u;

    for (;;) {
        unsigned idle = __ballot_sync(FULL, pid < 0);
        if (watchdog_tripped(iters, 1u << 22, w.counts)) break;
        idle = warp_refill(idle, TRACE4_REFILL_T, cursor, n, exhausted, pid, [&] {       // the ray lives at its queue position
            const float4 o = ro[pid];
            const float4 d = rd[pid];
            r = make_ray_fast(f3(o.x, o.y, o.z), f3(d.x, d.y, d.z), w.tmin, __float_as_int(o.w));
            best_t = ANY ? d.w - 1e-6f : w.tmax;                // shadow: dist - 1e-6 (Integrators.fs:44); closest: tMax (:108)
            best_slot = -1; pend = 0u; leafA = leafB = -1; h = 1u; depth = 0u;
            float e;
            local[0]++;
            const bool in = box_f(r, sc.root_min[0], sc.root_min[1], sc.root_min[2], sc.root_max[0], sc.root_max[1], sc.root_max[2], best_t, e);
            needPop = !in || sc.root_meta >= 0;     // nothing to descend into: the (empty) trail pop ends the ray
            if (in && sc.root_meta >= 0) leafA = sc.root_meta;
        });
        if (idle == FULL) { if (exhausted) break; continue; }

        // ---- node step(s) (lanes holding a node to visit and no parked leaves); TRACE4_NSTEP > 1 amortises the
        //      loop skeleton (ballots, vote, refill test) over several tree levels
#pragma unroll
        for (int rep = 0; rep < TRACE4_NSTEP; rep++)
        if (pid >= 0 && leafA < 0 && !needPop) {
            const PairF *pp = sc.pairs + h;
            const float4 q0 = ldg4(&pp->q0), q1 = ldg4(&pp->q1), q2 = ldg4(&pp->q2), q3 = ldg4(&pp->q3);
            local[0] += 2;
            const int metaL = __float_as_int(q3.x), metaR = __float_as_int(q3.y);
            float eL, eR;
            const bool hitL = box_f(r, q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, best_t, eL);
            const bool hitR = box_f(r, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w, best_t, eR);
            const bool rFirst = eR < eL;
            const bool lfL = hitL & (metaL >= 0), lfR = hitR & (metaR >= 0);
            const bool inL = hitL & (metaL < 0), inR = hitR & (metaR < 0);
            leafA = lfL ? ((lfR & rFirst) ? metaR : metaL) : (lfR ? metaR : -1);
            leafB = (lfL & lfR) ? (rFirst ? metaL : metaR) : -1;
            eB = rFirst ? eL : eR;
            const bool both = inL & inR;
            const bool rNear = inR & (!inL | rFirst);
            depth += (inL | inR) ? 1u : 0u;
            if (both) {
                pend |= 1u << depth;
                if (!ANY) lvl_entry[depth * FAST_BLOCK] = rNear ? eL : eR;
            }
            needPop = !(inL | inR);
            h = needPop ? h : (2u * h + (rNear ? 1u : 0u));
        }
        // ---- leaf phase by vote
        bool finished = false;
        if (leaf_vote(__ballot_sync(FULL, pid >= 0 && leafA >= 0), idle, TRACE4_LEAF_T)) {
            if (pid >= 0 && leafA >= 0) {
                bool found = leaf_f3<true, BIG>(sc, r, leafA, best_t, best_slot, local);
                if (leafB >= 0 && !(ANY && found) && eB <= best_t) found |= leaf_f3<true, BIG>(sc, r, leafB, best_t, best_slot, local);
                leafA = leafB = -1;
                if (ANY && found) finished = true;
            }
        }
        // ---- pop the deepest deferred sibling that can still beat the best hit
        if (pid >= 0 && needPop && leafA < 0 && !finished) {
            for (;;) {
                if (pend == 0u) { finished = true; break; }
                const unsigned b = 31u - __clz(pend);
                pend ^= 1u << b;
                if (ANY || lvl_entry[b * FAST_BLOCK] <= best_t) {
                    h = (h >> (depth - b)) ^ 1u;
                    depth = b;
                    needPop = false;
                    break;
                }
            }
        }
        if (finished) {
            if (!ANY) w.hit[pid] = make_float2(best_t, __int_as_float(best_slot));
            else if (best_slot < 0) { const float4 c = w.sh_c[pid]; float4 *ap = w.rad + __float_as_int(c.w); float4 a = *ap; a.x += c.x; a.y += c.y; a.z += c.z; *ap = a; }
            pid = -1;
        }
    }
    for (int k = 0; k < 3; k++) if (local[k]) atomicAdd(&ctr->v[ANY ? 1 : 0][k], local[k]);
}


// ---------------------------------------------------------------- own tree: SAH, four children per record, child links
// Same warp organisation as k_f_trace4 (ray replacement, two node steps per iteration, vote-postponed
// leaves), with a sorted 4-wide node step over the library's own binned-SAH tree (SceneF.own_tree, built by
// flatten_fast_own in mfx_host.cpp).  The tree is not heap-shaped, so the deferred hits go to a real stack; its layout,
// the child order (sort4), push, pop and launch geometry are shared with k_h_trace (mfx_fast_dev.cuh), like the ray
// replacement, leaf vote and watchdog of all three persistent-warp kernels.
// MFX_SKY_TRACER, late bounces (TAIL): the lane that finishes a closest-hit query shades it on the spot (one level of
// GetColor: sky_scatter_f, the function k_f_shade_sky calls too -- NOINLINE, so both run the same machine code and a
// frame does not depend on which of them shaded a vertex) and carries the scattered ray on until the path ends.  One
// launch takes every path still alive after bounce `MFX_SKY_TAIL` to the depth limit of 50 instead of two launches
// per bounce whose cost is launch latency (profiles/: ~30 us per bounce for a handful of rays), and the host never
// looks at a queue size in the middle of a Sample.
struct SkyCtx {
    const SlotF *slots; const float4 *slot_nrm; const MatF *mats; const float *perlin_rf; const int *perlin_perm;
    TileMap tm; int width, pix0, npix, s0; uint32_t k0, k1;
};
template <bool DIRECT>
__device__ bool sky_scatter_f(const SkyCtx &c, int k, int pid, int fs, float t, F3 o, F3 d, float4 &thr, float4 &st_o, float4 &st_d);

// Refill batches of 16 lanes, a leaf vote of 10 lanes, two node steps per iteration and one parked leaf per lane (the
// second nearest hit goes to the stack like any other) measured best in round 2 (profiles/); refill batches of 20 / 24 /
// 28 / 32 lanes (more sector sharing near the root, more idle lanes) measured -3 / -10 / -18 / -30 % on C2.
constexpr int TRACE6_REFILL_T = 16, TRACE6_LEAF_T = 10, TRACE6_NSTEP = 2;
template <bool ANY, bool BIG, int MINB, bool COUNT, bool TAIL = false>
__global__ void __launch_bounds__(FAST_BLOCK, MINB) k_f_trace6(SceneF sc, WaveF w, int bounce, TravCounters *ctr, SkyCtx sky)
{
    extern __shared__ uint2 s_stack[];              // [stack_smem][FAST_BLOCK]
    uint2 *my_stack = s_stack + threadIdx.x;
    const int S = sc.stack_smem;
    uint2 *my_spill = sc.stack_spill + ((size_t)blockIdx.x * FAST_BLOCK + threadIdx.x);
    const size_t spill_stride = (size_t)sc.spill_threads;
    const unsigned FULL = 0xffffffffu;
    const int n = ANY ? w.counts[CNT_SH(bounce)] : w.counts[bounce];
    const float4 *ro = ANY ? w.sh_o : w.ray_o[bounce & 1], *rd = ANY ? w.sh_d : w.ray_d[bounce & 1];
    int *cursor = &w.counts[ANY ? CUR_SH(bounce) : CUR_EXT(bounce)];
    const bool cam0 = !ANY && bounce == 0 && w.cam_origin;      // primary rays of a pinhole frame: the origin is a constant

    int pid = -1;
    RayF r;
    float best_t = 0.f; int best_slot = -1;
    int node = 0, sp = 0;                           // current record, stack height
    bool needPop = false;
    int leafA = -1;
    bool exhausted = false;
    unsigned iters = 0u;
    unsigned long long local[3] = { 0ull, 0ull, 0ull };   // COUNT: 128 B records fetched, triangle tests, sphere tests
    int path = -1, bnc = bounce, traced_on = 0;     // TAIL: path id, current bounce of the lane's path, rays traced beyond the queue's own
    float4 thr = make_float4(1.f, 1.f, 1.f, 0.f);   // TAIL: product of the attenuations so far

    for (;;) {
        unsigned idle = __ballot_sync(FULL, pid < 0);
        if (watchdog_tripped(iters, TAIL ? (1u << 26) : (1u << 22), w.counts)) break;
        idle = warp_refill(idle, TRACE6_REFILL_T, cursor, n, exhausted, pid, [&] {       // the ray lives at its queue position
            float4 o = make_float4(sc.cam.pos[0], sc.cam.pos[1], sc.cam.pos[2], __int_as_float(-1));
            if (!cam0) o = ro[pid];
            const float4 d = rd[pid];
            r = make_ray_fast(f3(o.x, o.y, o.z), f3(d.x, d.y, d.z), w.tmin, __float_as_int(o.w));
            best_t = ANY ? d.w - 1e-6f : w.tmax;                // shadow: dist - 1e-6 (Integrators.fs:44); closest: tMax (:108)
            best_slot = -1; sp = 0; leafA = -1; node = 0; needPop = false;
            if (TAIL) { path = __float_as_int(d.w); bnc = bounce; thr = w.thr[bounce & 1][pid]; }
        });
        if (idle == FULL) { if (exhausted) break; continue; }

#pragma unroll
        for (int rep = 0; rep < TRACE6_NSTEP; rep++)
        if (pid >= 0 && leafA < 0 && !needPop) {
            if (COUNT) local[0]++;
            const QuadF *qp = sc.quads + node;
            float4 lox, hix, loy, hiy, loz, hiz, m4, pad4;
            unsigned key[4];
            ldg8(&qp->lox, lox, hix); ldg8(&qp->loy, loy, hiy); ldg8(&qp->loz, loz, hiz); ldg8(&qp->meta, m4, pad4);
#define QUAD_SLOT(S_, C)                                                                                             \
            {                                                                                                        \
                const float x0 = fmaf(lox.C, r.idir.x, -r.ood.x), x1 = fmaf(hix.C, r.idir.x, -r.ood.x);              \
                const float y0 = fmaf(loy.C, r.idir.y, -r.ood.y), y1 = fmaf(hiy.C, r.idir.y, -r.ood.y);              \
                const float z0 = fmaf(loz.C, r.idir.z, -r.ood.z), z1 = fmaf(hiz.C, r.idir.z, -r.ood.z);              \
                const float tn = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fmaxf(fminf(z0, z1), r.tmin));           \
                const float tf = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fminf(fmaxf(z0, z1), best_t));           \
                const int mt = __float_as_int(m4.C);                                                                 \
                /* closest hit: nearest child first.  Shadow query: FARTHEST first -- any hit will do, the ray starts   \
                   inside the geometry it leaves (an occluded ray from the unlit side of a mesh walks the whole         \
                   interior nearest-first) and ends in the open near the light: tools/own_tree_sim.cpp, DESIGN.md 7.  \
                   Keys stay below KEY_INF (tn is finite and >= tMin > 0). */                                          \
                const unsigned ord = ANY ? (0x7f7ffff8u - (__float_as_uint(tn) & ~7u)) : (__float_as_uint(tn) & ~7u);   \
                key[S_] = (tn <= tf && mt != MFX_QUAD_EMPTY) ? (ord | (mt >= 0 ? 4u : 0u) | (unsigned)S_) : KEY_INF;   \
            }
            QUAD_SLOT(0, x) QUAD_SLOT(1, y) QUAD_SLOT(2, z) QUAD_SLOT(3, w)
#undef QUAD_SLOT
            unsigned k0, k1, k2, k3;
            sort4(key, k0, k1, k2, k3);
            const bool any0 = k0 != KEY_INF;
            const bool leaf0 = any0 && (k0 & 4u);
            const int c0 = pick4(m4, k0 & 3u);
            leafA = leaf0 ? c0 : -1;
            sp = own_push(my_stack, my_spill, S, spill_stride, sp, k1, k2, k3, node, sc, w.counts);
            const bool descend = any0 && !leaf0;
            needPop = !descend;
            if (descend) node = ~c0;
            DBG_CHECK(!descend || (unsigned)node < (unsigned)sc.n_quads, w.counts);
            DBG_CHECK(leafA < 0 || ((leafA >> 3) >= 0 && (leafA >> 3) + (leafA & 7) <= sc.n_slots), w.counts);
        }
        bool finished = false;
        if (leaf_vote(__ballot_sync(FULL, pid >= 0 && leafA >= 0), idle, TRACE6_LEAF_T)) {
            if (pid >= 0 && leafA >= 0) {
                const bool found = leaf_f3<COUNT, BIG>(sc, r, leafA, best_t, best_slot, local);
                leafA = -1;
                if (ANY && found) finished = true;
            }
        }
        if (pid >= 0 && needPop && leafA < 0 && !finished) {
            const OwnPop p = own_pop<ANY>(my_stack, my_spill, S, spill_stride, sp, best_t, sc, w.counts);
            sp = p.sp;
            if (!p.found) finished = true;
            else if (p.leaf) leafA = p.link;
            else { node = ~p.link; needPop = false; }
        }
        if (TAIL && finished) {
            // GetColor's next level, here and now (RayTracing.fs:367-382): a miss ends the path with T * sky, a hit at the
            // depth limit or a failed scatter ends it black, anything else scatters and the lane traces on
            DBG_CHECK(path >= 0 && path < w.P && best_slot < sc.n_slots, w.counts);
            bool again = false;
            if (best_slot < 0) {
                const float ty = 0.5f * (r.d.y + 1.0f);
                w.rad[path] = make_float4(thr.x * ((1.f - ty) + ty * 0.5f), thr.y * ((1.f - ty) + ty * 0.7f), thr.z * ((1.f - ty) + ty), 0.f);
            } else if (bnc < sc.max_depth) {
                float4 so, sd;
                if (sky_scatter_f<true>(sky, bnc, path, best_slot, best_t, r.o, r.d, thr, so, sd)) {
                    r = make_ray_fast(f3(so.x, so.y, so.z), f3(sd.x, sd.y, sd.z), w.tmin, __float_as_int(so.w));
                    best_t = w.tmax; best_slot = -1; sp = 0; leafA = -1; node = 0; needPop = false;
                    bnc++; traced_on++; again = true;
                }
            }
            if (!again) pid = -1;
        } else
        if (finished) {
            DBG_CHECK(pid >= 0 && pid < w.P && best_slot < sc.n_slots, w.counts);
            if (!ANY) w.hit[pid] = make_float2(best_t, __int_as_float(best_slot));
            else if (best_slot < 0) {
                const float4 c = w.sh_c[pid];
                DBG_CHECK(__float_as_int(c.w) >= 0 && __float_as_int(c.w) < w.P, w.counts);
                float4 *ap = w.rad + __float_as_int(c.w); float4 a = *ap; a.x += c.x; a.y += c.y; a.z += c.z; *ap = a;
            }
            pid = -1;
        }
    }
    if (COUNT) { for (int j = 0; j < 3; j++) if (local[j]) atomicAdd(&ctr->v[ANY ? 1 : 0][j], local[j]); }
    if (TAIL && traced_on) atomicAdd(&w.counts[bounce + 1], traced_on);     // the ray total sums counts[0..D]: the later bounces' rays land here
}

struct RngF { uint32_t pixel, sample, k0, k1; };

// GetRandomInUnitSphere (Material.fs:9-14) on the f32 view of the same Philox stream.
__device__ __forceinline__ F3 random_in_unit_sphere_f(F3 nm, const RngF &g, uint32_t dim)
{
    for (uint32_t it = 0; it < MFX_REJECTION_CAP; it++) {
        uint32_t o[4];
        philox4x32_10(g.pixel, g.sample, dim, it, g.k0, g.k1, o);
        const F3 p = f3(2.f * u32_to_unit_f32(o[0]) - 1.f, 2.f * u32_to_unit_f32(o[1]) - 1.f, 2.f * u32_to_unit_f32(o[2]) - 1.f);
        if (dot(p, p) < 1.0f && dot(nm, p) > 0.f) return p;
    }
    return nm;
}

// The same distribution without the loop (MFX_FAST_F32 default): GetRandomInUnitSphere(nm) is a uniform point of
// the half unit ball about nm, so its direction is uniform on the hemisphere and its radius is u^(1/3).  One Philox
// call feeds a whole vertex: o0,o1 -> direction, o2,o3 -> light point, spare low bits -> coin flip and radius.
// MFX_SAMPLE_REFERENCE_STREAM switches back to the reference's rejection loop on the exact mode's stream.
#define MFX_ITER_DIRECT 0xffffffffu
__device__ __forceinline__ F3 uniform_hemisphere_f(F3 nm, uint32_t a, uint32_t b)
{
    const float z = 1.f - 2.f * u32_to_unit_f32(a);
    const float r = sqrtf(fmaxf(0.f, 1.f - z * z));
    float sn, cs;
    __sincosf(6.283185307179586477f * u32_to_unit_f32(b), &sn, &cs);
    const F3 wdir = f3(r * cs, r * sn, z);
    return dot(nm, wdir) < 0.f ? -wdir : wdir;
}

__device__ __forceinline__ F3 tri_sample_f(const float *v0, const float *e1, const float *e2, float tu, float tv)
{
    float u = tu, v = tv;
    if (tu + tv > 1.f) { u = 1.f - tu; v = 1.f - tv; }
    const float sq = sqrtf(1.f - u);
    const float s1 = 1.f - sq, s2 = v * sq;
    return f3(v0[0] + e1[0] * s1 + e2[0] * s2, v0[1] + e1[1] * s1 + e2[1] * s2, v0[2] + e1[2] * s1 + e2[2] * s2);
}

__device__ __forceinline__ float fresnel_f(float eta_i, float eta_t, float cosi)    // Material.fs:74-96
{
    const float ei = cosi > 0.f ? eta_i : eta_t, et = cosi > 0.f ? eta_t : eta_i;
    const float sint = ei / et * sqrtf(fmaxf(0.f, 1.f - cosi * cosi));
    if (sint >= 1.f) return 1.f;
    const float cost = sqrtf(fmaxf(0.f, 1.f - sint * sint));
    const float ci = fabsf(cosi);
    const float rparl = ((et * ci) - (ei * cost)) / ((et * ci) + (ei * cost));
    const float rperp = ((ei * ci) - (et * cost)) / ((ei * ci) + (et * cost));
    return (rparl * rparl + rperp * rperp) * 0.5f;
}

// Shades vertex `bounce` of every path in the extend queue: BSDF/scatter sample, light sample,
// throughput update; compacts survivors into the next extend queue and the shadow queue with
// warp-aggregated appends.  Radiance bookkeeping (both integrators unrolled, see DESIGN.md):
//   mode 0 (Integrators.fs:136):  L += T * (l/pdf_li) * col ;  T *= col/pdf
//   mode 1 (PathTracer.fs:40-41): L += T * l * col          ;  T *= col * shadeFactor
#define SHADE_BLOCK 256
template <bool DIRECT>
__global__ void __launch_bounds__(SHADE_BLOCK, 4) k_f_shade(SceneF sc, WaveF w, TileMap tm, int pix0, int npix, int s0, int bounce, uint64_t seed)
{
    // Queue appends are aggregated per block: 5 000 resident warps hammering two counters with one atomic each per
    // iteration made the kernel wait on same-address atomics (72 % of its stall samples, profiles/); one atomic per
    // 256 paths and queue keeps the order inside a block.  Double-buffered by iteration parity: two barriers per pass.
    // The survivors' state is kept in registers across the barriers and written at the claimed positions, so the
    // next bounce's buffers are dense (see WaveF).
    __shared__ int s_cnt[2][2][SHADE_BLOCK / 32];
    __shared__ int s_base[2][2];
    const int n = w.counts[bounce];
    const int cur = bounce & 1, nxt = cur ^ 1;
    const float4 *in_o = w.ray_o[cur], *in_d = w.ray_d[cur], *in_thr = w.thr[cur];
    float4 *out_o = w.ray_o[nxt], *out_d = w.ray_d[nxt], *out_thr = w.thr[nxt];
    const int k = bounce;
    const bool last = (bounce >= sc.max_depth);
    const int nblock_iters = (n + SHADE_BLOCK - 1) / SHADE_BLOCK;
    const int stride = gridDim.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int it = blockIdx.x, par = 0;
    // the hit of the next iteration's entry is fetched one iteration ahead (the loads are consecutive now, this
    // only hides the first round trip)
    auto hit_at = [&](int iter) { const int i = iter * SHADE_BLOCK + threadIdx.x; return (iter < nblock_iters && i < n) ? w.hit[i] : make_float2(0.f, __int_as_float(-1)); };
    float2 hit_n = hit_at(it);
    for (; it < nblock_iters; it += stride, par ^= 1) {
        bool cont = false, shadow = false;
        const int i = it * SHADE_BLOCK + threadIdx.x;
        const float2 hr = hit_n;
        hit_n = hit_at(it + stride);
        float4 st_o = make_float4(0.f, 0.f, 0.f, 0.f), st_d = st_o, st_thr = st_o, st_shd = st_o, st_shc = st_o;
        if (i < n) {
            const int fs = __float_as_int(hr.y);
            if (fs >= 0) {
                const float t = hr.x;
                float4 o4 = make_float4(sc.cam.pos[0], sc.cam.pos[1], sc.cam.pos[2], __int_as_float(-1));
                if (!(bounce == 0 && w.cam_origin)) o4 = in_o[i];
                const float4 d4 = in_d[i];
                const int pid = __float_as_int(d4.w);                          // path id: RNG stream, slot of rad
                float4 thr = make_float4(1.f, 1.f, 1.f, 0.f);
                if (bounce > 0) thr = in_thr[i];
                const F3 o = f3(o4.x, o4.y, o4.z), d = f3(d4.x, d4.y, d4.z);
                const F3 point = o + d * t;
                const float4 sa = ldg4(&sc.slots[fs].a);
                const float4 sb = ldg4(&sc.slots[fs].b);
                const float4 nm4 = ldg4(&sc.slot_nrm[fs]);
                const int prim = __float_as_int(sb.w) & 0x3fffffff;
                F3 normal = f3(nm4.x, nm4.y, nm4.z);
                if (__float_as_int(sa.w) == 2) normal = normalize_f(point - f3(sa.x, sa.y, sa.z));
                else if (__float_as_int(sa.w) == 3) {       // big sphere: f64 centre (see leaf_f3)
                    const float4 sc4 = ldg4(&sc.slots[fs].c);
                    const double cx = __hiloint2double(__float_as_int(sb.y), __float_as_int(sb.x));
                    const double cy = __hiloint2double(__float_as_int(sc4.y), __float_as_int(sc4.x));
                    const double cz = __hiloint2double(__float_as_int(sc4.w), __float_as_int(sc4.z));
                    normal = normalize_f(f3((float)((double)point.x - cx), (float)((double)point.y - cy), (float)((double)point.z - cz)));
                }
                DBG_CHECK(fs < sc.n_slots && pid >= 0 && pid < w.P && (unsigned)__float_as_int(nm4.w) < (unsigned)sc.n_mats, w.counts);
                const MatF m = sc.mats[__float_as_int(nm4.w)];
                int sl, pl;
                path_split(tm, pid, npix, sl, pl);
                int pix, px, py;
                pixel_of(tm, sc.width, pix0 + pl, pix, px, py);
                DBG_CHECK(pix >= 0 && pix < sc.width * sc.height, w.counts);
                RngF g; g.pixel = (uint32_t)pix; g.sample = (uint32_t)(s0 + sl); g.k0 = (uint32_t)seed; g.k1 = (uint32_t)(seed >> 32);

                uint32_t dz[4] = { 0u, 0u, 0u, 0u };
                F3 hemi = normal;                          // DIRECT: unit vector, uniform on the hemisphere about `normal`
                if (DIRECT) {
                    philox4x32_10(g.pixel, g.sample, MFX_DIM_BSDF(k), MFX_ITER_DIRECT, g.k0, g.k1, dz);
                    hemi = uniform_hemisphere_f(normal, dz[0], dz[1]);
                }
                F3 wi; float cr, cg, cb; float sf = 1.f;   // col and the Shade factor applied to the continuation
                if (sc.mode == 0) {
                    const float z = (m.kind == 2) ? 0.f : 1.f;
                    wi = DIRECT ? hemi : normalize_f(random_in_unit_sphere_f(normal, g, MFX_DIM_BSDF(k)));
                    const float ei2 = 2.f * dot(normal, wi);                 // INVPI * a * ei * TwoPi
                    cr = z * m.albedo[0] * ei2; cg = z * m.albedo[1] * ei2; cb = z * m.albedo[2] * ei2;
                } else if (m.kind == 0) {
                    wi = DIRECT ? hemi : normalize_f(random_in_unit_sphere_f(normal, g, MFX_DIM_BSDF(k)));
                    const float ip = 0.318309886183790672f;
                    cr = m.albedo[0] * ip; cg = m.albedo[1] * ip; cb = m.albedo[2] * ip;
                    sf = 6.283185307179586477f * dot(normal, wi);            // Lambertian.Shade
                } else if (m.kind == 1) {
                    const float fuzz = fminf(m.fuzz, 1.f);
                    const F3 refl = d - normal * (2.f * dot(d, normal));
                    F3 ball;
                    if (DIRECT) {       // radius of a uniform ball point from the 24 spare low bits of o1..o3
                        const uint32_t rb = ((dz[1] & 0xffu) << 24) | ((dz[2] & 0xffu) << 16) | ((dz[3] & 0xffu) << 8);
                        ball = hemi * cbrtf(u32_to_unit_f32(rb));
                    } else ball = random_in_unit_sphere_f(normal, g, MFX_DIM_BSDF(k));
                    wi = normalize_f(refl + ball * fuzz);
                    cr = m.albedo[0]; cg = m.albedo[1]; cb = m.albedo[2];
                } else {
                    const F3 dir = -d;
                    const float cosi = dot(dir, normal);
                    const float ei = cosi > 0.f ? m.ei : m.et, et = cosi > 0.f ? m.et : m.ei;
                    const float r = ei / et;
                    const float dt = dot(normalize_f(dir), normal);
                    const float disc = 1.f - r * r * (1.f - dt * dt);
                    if (disc > 0.f) {
                        wi = (dir - normal * dt) * r - normal * sqrtf(disc);
                        const float F = fresnel_f(m.ei, m.et, cosi);
                        const float f = (et * et) / (ei * ei) * (1.f - F) / fabsf(dot(wi, normal));
                        cr = f * m.albedo[0]; cg = f * m.albedo[1]; cb = f * m.albedo[2];
                    } else {
                        wi = dir - normal * (2.f * dot(dir, normal));
                        cr = cg = cb = 0.f;
                    }
                }
                // light sample (Rect.fs:33-38, Trangle.fs:157-169, Light.fs:42-59)
                uint32_t lo4[4];
                if (DIRECT) { lo4[0] = dz[0] << 31; lo4[1] = dz[2]; lo4[2] = dz[3]; }     // coin = spare low bit of o0
                else philox4x32_10(g.pixel, g.sample, MFX_DIM_LIGHT(k), 0, g.k0, g.k1, lo4);
                const float tu = u32_to_unit_f32(lo4[1]), tv = u32_to_unit_f32(lo4[2]);
                // the coin uses the full 32-bit value so it matches the f64 stream's `s < 0.5`
                const F3 lp = (lo4[0] < 0x80000000u) ? tri_sample_f(sc.light.v0a, sc.light.e1a, sc.light.e2a, tu, tv)
                                                     : tri_sample_f(sc.light.v0b, sc.light.e1b, sc.light.e2b, tu, tv);
                const F3 toLight = lp - point;
                const float d2 = len2(toLight);
                const float dist = sqrtf(d2);
                const F3 unit = toLight * (1.f / dist);
                const float cos_o = dot(toLight, f3(sc.light.normal[0], sc.light.normal[1], sc.light.normal[2]));
                float lscale = 0.f;
                if (cos_o < 0.f) lscale = dot(unit, normal) * (fabsf(cos_o) * sc.light.area / d2);
                if (sc.mode == 0) lscale *= sc.light.inv_pdf;                // l / pdf_li
                st_shc = make_float4(thr.x * cr * lscale * sc.light.color[0], thr.y * cg * lscale * sc.light.color[1],
                                     thr.z * cb * lscale * sc.light.color[2], __int_as_float(pid));
                shadow = (st_shc.x != 0.f) || (st_shc.y != 0.f) || (st_shc.z != 0.f);
                thr.x *= cr * sf; thr.y *= cg * sf; thr.z *= cb * sf;
                cont = !last && ((thr.x != 0.f) || (thr.y != 0.f) || (thr.z != 0.f));
                // planar sources are never re-hit; spheres keep themselves as source (far root / none)
                st_o = make_float4(point.x, point.y, point.z, __int_as_float(prim));
                st_d = make_float4(wi.x, wi.y, wi.z, __int_as_float(pid));
                st_thr = thr;
                st_shd = make_float4(unit.x, unit.y, unit.z, dist);
            }
        }
        const unsigned mc = __ballot_sync(0xffffffffu, cont), ms = __ballot_sync(0xffffffffu, shadow);
        if (lane == 0) { s_cnt[par][0][warp] = __popc(mc); s_cnt[par][1][warp] = __popc(ms); }
        __syncthreads();
        if (threadIdx.x < 2) {
            int tot = 0;
            for (int j = 0; j < SHADE_BLOCK / 32; j++) { const int c = s_cnt[par][threadIdx.x][j]; s_cnt[par][threadIdx.x][j] = tot; tot += c; }
            int *counter = &w.counts[threadIdx.x == 0 ? bounce + 1 : MFX_MAX_VERTS + 2 + bounce];
            s_base[par][threadIdx.x] = tot ? atomicAdd(counter, tot) : 0;
        }
        __syncthreads();
        const unsigned below = (1u << lane) - 1u;
        if (cont) {
            const int pos = s_base[par][0] + s_cnt[par][0][warp] + __popc(mc & below);
            DBG_CHECK(pos >= 0 && pos < w.P, w.counts);
            out_o[pos] = st_o; out_d[pos] = st_d; out_thr[pos] = st_thr;
        }
        if (shadow) {
            const int pos = s_base[par][1] + s_cnt[par][1][warp] + __popc(ms & below);
            DBG_CHECK(pos >= 0 && pos < w.P, w.counts);
#ifdef MFX_DEBUG_CHECKS
            // the shadow kernel adds to rad[path] without an atomic: sound only while a path has at most ONE shadow ray in
            // flight per bounce -- every path stamps the bounce that queued its ray, a second stamp of the same bounce trips
            if (w.dbg_stamp) DBG_CHECK(atomicExch(&w.dbg_stamp[__float_as_int(st_shc.w)], bounce + 1) != bounce + 1, w.counts);
#endif
            w.sh_o[pos] = st_o; w.sh_d[pos] = st_shd; w.sh_c[pos] = st_shc;
        }
    }
}

// ---------------------------------------------------------------- MFX_SKY_TRACER shading
// One level of GetColor (RenderTest/Sample/RayTracing.fs:367-382) for every path in the extend queue, unrolled like
// the other integrators: T = product of the attenuations so far; a miss ends the path with rad = T * sky, a hit at
// the depth limit or a failed scatter ends it black, anything else scatters (Lambertian :282-290, Metal :291-299,
// Dielectric :300-325) and joins the next extend queue.  No light, no shadow queue.
// DIRECT (default): GetRandomInUnitSphere (:261-266, the whole ball) drawn without the loop -- uniform direction,
// radius u^(1/3) -- one Philox call per vertex feeds the ball and the dielectric coin.  MFX_SAMPLE_REFERENCE_STREAM
// runs the rejection loop on the exact mode's stream instead.
__device__ __forceinline__ F3 random_in_unit_ball_f(const RngF &g, uint32_t dim)
{
    for (uint32_t it = 0; it < MFX_REJECTION_CAP; it++) {
        uint32_t o[4];
        philox4x32_10(g.pixel, g.sample, dim, it, g.k0, g.k1, o);
        const F3 p = f3(2.f * u32_to_unit_f32(o[0]) - 1.f, 2.f * u32_to_unit_f32(o[1]) - 1.f, 2.f * u32_to_unit_f32(o[2]) - 1.f);
        if (dot(p, p) < 1.0f) return p;
    }
    return f3(0.f, 0.f, 0.f);
}

// One level of GetColor for a ray (o, d) that hit fast slot fs at distance t: scatter (Lambertian :282-290, Metal :291-299,
// Dielectric :300-325), attenuation into thr; true if the path goes on (st_o / st_d: its next ray, source primitive and
// path id in the w fields).  NOINLINE on purpose: see SkyCtx.
template <bool DIRECT>
__device__ __noinline__ bool sky_scatter_f(const SkyCtx &c, int k, int pid, int fs, float t, F3 o, F3 d, float4 &thr, float4 &st_o, float4 &st_d)
{
    const F3 point = o + d * t;
    const float4 sa = ldg4(&c.slots[fs].a);
    const float4 sb = ldg4(&c.slots[fs].b);
    const int prim = __float_as_int(sb.w) & 0x3fffffff;
    F3 normal;                                                         // (p - center) / radius, :198
    if (__float_as_int(sa.w) == 3) {                                   // big sphere: f64 centre (see leaf_f3)
        const float4 sc4 = ldg4(&c.slots[fs].c);
        const double cx = __hiloint2double(__float_as_int(sb.y), __float_as_int(sb.x));
        const double cy = __hiloint2double(__float_as_int(sc4.y), __float_as_int(sc4.x));
        const double cz = __hiloint2double(__float_as_int(sc4.w), __float_as_int(sc4.z));
        normal = normalize_f(f3((float)((double)point.x - cx), (float)((double)point.y - cy), (float)((double)point.z - cz)));
    } else normal = normalize_f(point - f3(sa.x, sa.y, sa.z));
    const MatF m = c.mats[__float_as_int(ldg4(&c.slot_nrm[fs]).w)];
    int sl, pl;
    path_split(c.tm, pid, c.npix, sl, pl);
    int pix, px, py;
    pixel_of(c.tm, c.width, c.pix0 + pl, pix, px, py);
    RngF g; g.pixel = (uint32_t)pix; g.sample = (uint32_t)(c.s0 + sl); g.k0 = c.k0; g.k1 = c.k1;
    uint32_t dz[4] = { 0u, 0u, 0u, 0u };
    if (DIRECT) philox4x32_10(g.pixel, g.sample, MFX_DIM_BSDF(k), MFX_ITER_DIRECT, g.k0, g.k1, dz);
    F3 wi, att;
    bool ok = true;
    if (m.kind == 3) {                                                 // Dielectric
        const float dn = dot(d, normal);
        const F3 reflected = d - normal * (2.f * dn);
        const F3 outward = dn > 0.f ? -normal : normal;
        const float nint = dn > 0.f ? m.ei : 1.f / m.ei;
        const float cosine = dn > 0.f ? m.ei * dn : -dn;
        const float dt = dot(d, outward);
        const float disc = 1.f - nint * nint * (1.f - dt * dt);
        float reflect_prob = 1.f;
        F3 ref_dir = reflected;
        if (disc > 0.f) {
            ref_dir = (d - outward * dt) * nint - outward * sqrtf(disc);
            const float r0 = (1.f - m.ei) / (1.f + m.ei), r1 = r0 * r0;
            const float x = 1.f - cosine, x2 = x * x;
            reflect_prob = r1 + (1.f - r1) * (x2 * x2 * x);
        }
        uint32_t coin = dz[3];
        if (!DIRECT) { uint32_t c4[4]; philox4x32_10(g.pixel, g.sample, MFX_DIM_LIGHT(k), 0, g.k0, g.k1, c4); coin = c4[0]; }
        // the coin uses the full 32-bit value like the f64 stream's `NextDouble() < reflect_prob`
        wi = normalize_f(((double)coin * (1.0 / 4294967296.0) < (double)reflect_prob) ? reflected : ref_dir);
        att = f3(1.f, 1.f, 1.f);
    } else {
        F3 ball;
        if (DIRECT) {
            const float z = 1.f - 2.f * u32_to_unit_f32(dz[0]);
            const float r = sqrtf(fmaxf(0.f, 1.f - z * z));
            float sn, cs;
            __sincosf(6.283185307179586477f * u32_to_unit_f32(dz[1]), &sn, &cs);
            ball = f3(r * cs, r * sn, z) * cbrtf(u32_to_unit_f32(dz[2]));
        } else ball = random_in_unit_ball_f(g, MFX_DIM_BSDF(k));
        if (m.kind == 1) {                                             // Metal
            const float fuzz = fminf(m.fuzz, 1.f);
            wi = normalize_f(d - normal * (2.f * dot(d, normal)) + ball * fuzz);
            att = f3(m.albedo[0], m.albedo[1], m.albedo[2]);
            ok = dot(wi, normal) > 0.f;
        } else {                                                       // Lambertian over a texture (:50-61, :86-99)
            wi = normalize_f(normal + ball);
            att = f3(m.albedo[0], m.albedo[1], m.albedo[2]);
            if (m.kind == 4) {
                if (sinf(10.f * point.x) * sinf(10.f * point.y) * sinf(10.f * point.z) < 0.f) att = f3(m.fuzz, m.ei, m.et);
            } else if (m.kind == 5) {
                const int ia = (int)(4.f * point.x) & 255, ib = (int)(4.f * point.y) & 255, ic = (int)(4.f * point.z) & 255;
                const float nz = __ldg(&c.perlin_rf[__ldg(&c.perlin_perm[ia]) ^ __ldg(&c.perlin_perm[256 + ib]) ^ __ldg(&c.perlin_perm[512 + ic])]);
                att = f3(nz, nz, nz);
            }
        }
    }
    thr.x *= att.x; thr.y *= att.y; thr.z *= att.z;
    const bool cont = ok && ((thr.x != 0.f) || (thr.y != 0.f) || (thr.z != 0.f));
    st_o = make_float4(point.x, point.y, point.z, __int_as_float(prim));
    st_d = make_float4(wi.x, wi.y, wi.z, __int_as_float(pid));
    return cont;
}

template <bool DIRECT>
__global__ void __launch_bounds__(SHADE_BLOCK, 4) k_f_shade_sky(SceneF sc, WaveF w, TileMap tm, int pix0, int npix, int s0, int bounce, uint64_t seed)
{
    __shared__ int s_cnt[2][SHADE_BLOCK / 32];
    __shared__ int s_base[2];
    const int n = w.counts[bounce];
    const int cur = bounce & 1, nxt = cur ^ 1;
    const int k = bounce;
    const bool last = (bounce >= sc.max_depth);          // `depth < 50`, :373
    const int nblock_iters = (n + SHADE_BLOCK - 1) / SHADE_BLOCK;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const SkyCtx ctx{ sc.slots, sc.slot_nrm, sc.mats, sc.perlin_rf, sc.perlin_perm, tm, sc.width, pix0, npix, s0, (uint32_t)seed, (uint32_t)(seed >> 32) };
    int par = 0;
    for (int it = blockIdx.x; it < nblock_iters; it += gridDim.x, par ^= 1) {
        const int i = it * SHADE_BLOCK + threadIdx.x;
        bool cont = false;
        float4 st_o = make_float4(0.f, 0.f, 0.f, 0.f), st_d = st_o, st_thr = st_o;
        if (i < n) {
            const float2 hr = w.hit[i];
            const int fs = __float_as_int(hr.y);
            const float4 d4 = w.ray_d[cur][i];
            const int pid = __float_as_int(d4.w);                                  // path id: RNG stream, slot of rad
            float4 thr = make_float4(1.f, 1.f, 1.f, 0.f);
            if (bounce > 0) thr = w.thr[cur][i];
            const F3 d = f3(d4.x, d4.y, d4.z);
            if (fs < 0) {
                const float t = 0.5f * (d.y + 1.0f);                               // :378-381 (d is unit)
                w.rad[pid] = make_float4(thr.x * ((1.f - t) + t * 0.5f), thr.y * ((1.f - t) + t * 0.7f), thr.z * ((1.f - t) + t), 0.f);
            } else if (!last) {
                float4 o4 = make_float4(sc.cam.pos[0], sc.cam.pos[1], sc.cam.pos[2], __int_as_float(-1));
                if (!(bounce == 0 && w.cam_origin)) o4 = w.ray_o[cur][i];
                cont = sky_scatter_f<DIRECT>(ctx, k, pid, fs, hr.x, f3(o4.x, o4.y, o4.z), d, thr, st_o, st_d);
                st_thr = thr;
            }
        }
        const unsigned mc = __ballot_sync(0xffffffffu, cont);
        if (lane == 0) s_cnt[par][warp] = __popc(mc);
        __syncthreads();
        if (threadIdx.x == 0) {
            int tot = 0;
            for (int j = 0; j < SHADE_BLOCK / 32; j++) { const int c = s_cnt[par][j]; s_cnt[par][j] = tot; tot += c; }
            s_base[par] = tot ? atomicAdd(&w.counts[bounce + 1], tot) : 0;
        }
        __syncthreads();
        if (cont) {
            const int pos = s_base[par] + s_cnt[par][warp] + __popc(mc & ((1u << lane) - 1u));
            w.ray_o[nxt][pos] = st_o; w.ray_d[nxt][pos] = st_d; w.thr[nxt][pos] = st_thr;
        }
    }
}

__global__ void __launch_bounds__(256) k_f_resolve(SceneF sc, WaveF w, TileMap tm, int pix0, int npix, int S, double *pixsum)
{
    for (int pl = blockIdx.x * blockDim.x + threadIdx.x; pl < npix; pl += gridDim.x * blockDim.x) {
        int pix, px, py;
        pixel_of(tm, sc.width, pix0 + pl, pix, px, py);
        // f64 running sums in absolute sample order: the frame does not depend on how spp was cut into waves
        // (world size, MFX_WAVE_PATHS, the out-of-memory halving)
        double *p = pixsum + 4 * (size_t)pix;
        double r = p[0], g = p[1], b = p[2];
        for (int sl = 0; sl < S; sl++) {
            const float4 a = w.rad[path_join(tm, sl, pl, npix)];
            r += (double)a.x; g += (double)a.y; b += (double)a.z;
        }
        p[0] = r; p[1] = g; p[2] = b; p[3] = 1.0;
    }
}

// Finer seams (Bvh.Hit, GetRay + Hit) routed through the PRODUCTION traversal kernel: rays are written
// into the wave's queues, traced by k_f_trace6, and read back.  src (nullptr: none): per ray, the id the fast slots carry
// for the primitive it starts on, or -1 -- what the shade kernels write into ray_o.w / sh_o.w.
__global__ void __launch_bounds__(256) k_f_seam_setup(SceneF sc, WaveF w, int n, const double *o, const double *d, const double *uv,
                                                      const int *src, long long first, float tmax, int any_hit)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const long long r = first + i;
        const int sp = src ? src[r] : -1;
        F3 oo, dd;
        if (d) {
            oo = f3((float)o[3 * r], (float)o[3 * r + 1], (float)o[3 * r + 2]);
            dd = f3((float)d[3 * r], (float)d[3 * r + 1], (float)d[3 * r + 2]);
            if (sc.mode == MFX_MODE_SKY) {      // Ray(origin, direc) normalises (RayTracing.fs:14-16)
                const double l = sqrt(d[3 * r] * d[3 * r] + d[3 * r + 1] * d[3 * r + 1] + d[3 * r + 2] * d[3 * r + 2]);
                dd = f3((float)(d[3 * r] / l), (float)(d[3 * r + 1] / l), (float)(d[3 * r + 2] / l));
            }
        } else {
            double u, v;
            if (uv) { u = uv[2 * r]; v = uv[2 * r + 1]; }
            else {
                const int j = (int)(r / sc.width), ii = (int)(r - (long long)j * sc.width);
                u = ((double)ii + 0.5) / (double)sc.width;
                v = ((double)j + 0.5) / (double)sc.height;
            }
            oo = f3(sc.cam.pos[0], sc.cam.pos[1], sc.cam.pos[2]);
            dd = camera_dir_f64(sc.camx, u, v);
        }
        w.ray_o[0][i] = make_float4(oo.x, oo.y, oo.z, __int_as_float(sp));
        w.ray_d[0][i] = make_float4(dd.x, dd.y, dd.z, __int_as_float(i));   // tMax of the closest query is w.tmax
        w.sh_o[i] = make_float4(oo.x, oo.y, oo.z, __int_as_float(sp));
        w.sh_d[i] = make_float4(dd.x, dd.y, dd.z, tmax + 1e-6f);      // the shadow kernel subtracts 1e-6 (Integrators.fs:44)
        w.sh_c[i] = make_float4(1.f, 0.f, 0.f, __int_as_float(i));    // unoccluded rays add this to rad[i]
        w.rad[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        w.hit[i] = make_float2(0.f, __int_as_float(-1));
        if (i == 0) { w.counts[0] = any_hit ? 0 : n; w.counts[CNT_SH(0)] = any_hit ? n : 0; }
    }
}

__global__ void __launch_bounds__(256) k_f_seam_read(SceneF sc, WaveF w, int n, long long first, int any_hit, int *prim, int *sub, double *t)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const long long r = first + i;
        if (any_hit) {                          // only occluded / clear is meaningful
            prim[r] = (w.rad[i].x == 0.f) ? 0 : -1;
            if (sub) sub[r] = 0;
            t[r] = 0.;
            continue;
        }
        const float2 h = w.hit[i];
        const int slot = __float_as_int(h.y);
        if (slot < 0) { prim[r] = -1; if (sub) sub[r] = 0; t[r] = 0.; }
        else {
            const int ps = __float_as_int(sc.slots[slot].b.w);
            prim[r] = sc.ref_id ? sc.ref_id[ps & 0x3fffffff] : (ps & 0x3fffffff);
            if (sub) sub[r] = (ps >> 30) & 1;
            t[r] = (double)h.x;
        }
    }
}

// ---------------------------------------------------------------- utility kernels
__global__ void k_accum_totals(const int *counts, int ext_lo, int ext_n, int sh_lo, int sh_n, unsigned long long *totals)
{
    unsigned long long e = 0, s = 0;
    for (int i = 0; i < ext_n; i++) e += (unsigned)counts[ext_lo + i];
    for (int i = 0; i < sh_n; i++) s += (unsigned)counts[sh_lo + i];
    totals[0] += e; totals[1] += s; totals[2] += (unsigned)counts[0];
    totals[3] += (unsigned)counts[MFX_COUNTS_LEN - 1];      // traversal watchdog trips
    totals[5] += (unsigned)counts[MFX_DBG_SLOT];            // violations counted by a debug build (MFX_DEBUG_CHECKS)
}

// The film kernels work on the pixels `tm` owns (pixel_of): a device of mfx_multi_film_* touches its own column stripes
// only, the one-GPU film passes one stripe as wide as the frame.  Color[w,h] buffers are x-major (x*H+y), RGBA8 row-major.

// Film.AddSample (Film.fs:18-23): c = sum + frame; sum <- c; target <- c / frameCount
__global__ void __launch_bounds__(256) k_film_add(TileMap tm, int width, double *sum, const double *frame, double *target, double fc)
{
    for (int pl = blockIdx.x * blockDim.x + threadIdx.x; pl < tm.n_pix; pl += gridDim.x * blockDim.x) {
        int pix, x, y;
        pixel_of(tm, width, pl, pix, x, y);
        const size_t p = (size_t)x * tm.height + y;
        for (int c = 0; c < 3; c++) {
            const double v = sum[4 * p + c] + frame[4 * p + c];
            sum[4 * p + c] = v;
            target[4 * p + c] = v / fc;
        }
        const double a = sum[4 * p + 3] + frame[4 * p + 3];
        sum[4 * p + 3] = a < 1.0 ? a : 1.0;
        target[4 * p + 3] = 1.0;
    }
}

__device__ __forceinline__ double clamp01(double x) { return x < 0. ? 0. : (x > 1. ? 1. : x); }

// ACESFilmToneMapping + sqrt + int(255.99 c) (Scene.fs:273-289,315-330).  target is Color[w,h]
// x-major; out is RGBA8 at x*4 + y*width*4.  f64 with explicit non-fused operations.
__global__ void __launch_bounds__(256) k_film_tonemap(TileMap tm, int width, const double *target, uint8_t *rgba8)
{
    for (int pl = blockIdx.x * blockDim.x + threadIdx.x; pl < tm.n_pix; pl += gridDim.x * blockDim.x) {
        int pix, x, y;
        pixel_of(tm, width, pl, pix, x, y);
        const double *px = target + ((size_t)x * tm.height + y) * 4;
        uint8_t out[4];
        for (int c = 0; c < 3; c++) {
            const double v = px[c];
            const double num = __dmul_rn(v, __dadd_rn(__dmul_rn(2.51, v), 0.03));
            const double den = __dadd_rn(__dmul_rn(v, __dadd_rn(__dmul_rn(2.43, v), 0.59)), 0.14);
            const double q = sqrt(clamp01(num / den));
            out[c] = (uint8_t)(int)__dmul_rn(255.99, q);
        }
        out[3] = 255;
        *reinterpret_cast<uchar4 *>(rgba8 + 4 * (size_t)pix) = make_uchar4(out[0], out[1], out[2], out[3]);
    }
}

// The sphere sample's display transform (RenderTest/Sample/RayTracing.fs:456-460): sqrt, int(255.99 c), and
// screen[i, (ny-1)-j]: row j of the texture (v grows upwards from lowerLeftCorner) lands on screen row ny-1-j.  The flip
// keeps the column, so a device's stripes of the screen come from its own stripes of the texture.
__global__ void __launch_bounds__(256) k_film_display_sky(TileMap tm, int width, const double *target, uint8_t *rgba8)
{
    for (int pl = blockIdx.x * blockDim.x + threadIdx.x; pl < tm.n_pix; pl += gridDim.x * blockDim.x) {
        int pix, x, y;
        pixel_of(tm, width, pl, pix, x, y);
        const double *px = target + ((size_t)x * tm.height + (tm.height - 1 - y)) * 4;
        uint8_t out[3];
        for (int c = 0; c < 3; c++) {
            const double v = __dmul_rn(255.99, sqrt(px[c]));
            out[c] = (v == v) ? (uint8_t)(int)v : 0;
        }
        *reinterpret_cast<uchar4 *>(rgba8 + 4 * (size_t)pix) = make_uchar4(out[0], out[1], out[2], 255);
    }
}

// ---------------------------------------------------------------- launchers
void mfx_f_raygen(const LaunchCfg &c, const SceneF &sc, const WaveF &w, TileMap tm, int pix0, int npix, int s0, int S, uint64_t seed)
{
    k_f_raygen<<<persistent_blocks(k_f_raygen, 256, c.blocks), 256, 0, c.stream>>>(sc, w, tm, pix0, npix, s0, S, seed);
}
template <bool ANY, bool BIG>
static void launch_trace4(const LaunchCfg &c, const SceneF &sc, const WaveF &w, int bounce, TravCounters *ctr)
{
    const size_t smem = ANY ? 0 : (size_t)sc.levels * FAST_BLOCK * sizeof(float);
    k_f_trace4<ANY, BIG><<<persistent_blocks(k_f_trace4<ANY, BIG>, FAST_BLOCK, c.blocks, smem), FAST_BLOCK, smem, c.stream>>>(sc, w, bounce, ctr);
}
template <bool ANY, bool BIG, int MB, bool CNT, bool TAIL = false>
static void launch_trace6(const LaunchCfg &c, const SceneF &sc, const WaveF &w, int bounce, TravCounters *ctr, const SkyCtx &sky = SkyCtx{})
{
    k_f_trace6<ANY, BIG, MB, CNT, TAIL><<<own_tree_blocks(k_f_trace6<ANY, BIG, MB, CNT, TAIL>, c, sc), FAST_BLOCK, own_stack_smem(sc), c.stream>>>(sc, w, bounce, ctr, sky);
}
// The layout decides the kernel: the reference tree is passed for the instrumented counting runs (the algorithmic record
// counts of the roofline are defined on the reference's binary tree) and takes k_f_trace4; the library's SAH tree takes
// k_f_trace6, instrumented when counters were asked for (MFX_SAMPLE_COUNT_OWN_TREE).  Scenes without a big (f64) sphere
// get the kernels compiled without that branch.
template <bool ANY>
static void launch_trace(const LaunchCfg &c, const SceneF &sc, const WaveF &w, int bounce, TravCounters *ctr)
{
    const bool big = sc.has_big_sphere != 0;
    if (!sc.own_tree) { if (big) launch_trace4<ANY, true>(c, sc, w, bounce, ctr); else launch_trace4<ANY, false>(c, sc, w, bounce, ctr); }
    else if (ctr) { if (big) launch_trace6<ANY, true, 1, true>(c, sc, w, bounce, ctr); else launch_trace6<ANY, false, 1, true>(c, sc, w, bounce, ctr); }
    else if (big) launch_trace6<ANY, true, 8, false>(c, sc, w, bounce, nullptr);        // 8 blocks/SM: 64 registers
    else launch_trace6<ANY, false, 8, false>(c, sc, w, bounce, nullptr);
}
void mfx_f_extend(const LaunchCfg &c, const SceneF &sc, const WaveF &w, int bounce, TravCounters *ctr)
{
    launch_trace<false>(c, sc, w, bounce, ctr);
}
// MFX_SKY_TRACER: every path in the extend queue of `bounce` traced AND shaded to its end in one launch (k_f_trace6<TAIL>)
void mfx_f_sky_tail(const LaunchCfg &c, const SceneF &sc, const WaveF &w, TileMap tm, int pix0, int npix, int s0, int bounce, uint64_t seed)
{
    const SkyCtx sky{ sc.slots, sc.slot_nrm, sc.mats, sc.perlin_rf, sc.perlin_perm, tm, sc.width, pix0, npix, s0, (uint32_t)seed, (uint32_t)(seed >> 32) };
    if (sc.has_big_sphere) launch_trace6<false, true, 4, false, true>(c, sc, w, bounce, nullptr, sky);
    else launch_trace6<false, false, 4, false, true>(c, sc, w, bounce, nullptr, sky);
}
void mfx_f_shade(const LaunchCfg &c, const SceneF &sc, const WaveF &w, TileMap tm, int pix0, int npix, int s0, int bounce, uint64_t seed)
{
    if (c.reference_stream) k_f_shade<false><<<persistent_blocks(k_f_shade<false>, SHADE_BLOCK, c.blocks), SHADE_BLOCK, 0, c.stream>>>(sc, w, tm, pix0, npix, s0, bounce, seed);
    else k_f_shade<true><<<persistent_blocks(k_f_shade<true>, SHADE_BLOCK, c.blocks), SHADE_BLOCK, 0, c.stream>>>(sc, w, tm, pix0, npix, s0, bounce, seed);
}
void mfx_f_shade_sky(const LaunchCfg &c, const SceneF &sc, const WaveF &w, TileMap tm, int pix0, int npix, int s0, int bounce, uint64_t seed)
{
    int blocks = c.reference_stream ? persistent_blocks(k_f_shade_sky<false>, SHADE_BLOCK, c.blocks) : persistent_blocks(k_f_shade_sky<true>, SHADE_BLOCK, c.blocks);
    if (c.max_items > 0) blocks = std::max(1, std::min(blocks, (c.max_items + SHADE_BLOCK - 1) / SHADE_BLOCK));
    if (c.reference_stream) k_f_shade_sky<false><<<blocks, SHADE_BLOCK, 0, c.stream>>>(sc, w, tm, pix0, npix, s0, bounce, seed);
    else k_f_shade_sky<true><<<blocks, SHADE_BLOCK, 0, c.stream>>>(sc, w, tm, pix0, npix, s0, bounce, seed);
}
void mfx_f_shadow(const LaunchCfg &c, const SceneF &sc, const WaveF &w, int bounce, TravCounters *ctr)
{
    launch_trace<true>(c, sc, w, bounce, ctr);
}
void mfx_f_resolve(const LaunchCfg &c, const SceneF &sc, const WaveF &w, TileMap tm, int pix0, int npix, int S, double *pixsum)
{
    k_f_resolve<<<persistent_blocks(k_f_resolve, 256, c.blocks), 256, 0, c.stream>>>(sc, w, tm, pix0, npix, S, pixsum);
}
void mfx_f_seam_setup(const LaunchCfg &c, const SceneF &sc, const WaveF &w, int n, const double *o, const double *d, const double *uv,
                      const int *src, long long first, float tmax, int any_hit)
{
    k_f_seam_setup<<<persistent_blocks(k_f_seam_setup, 256, c.blocks), 256, 0, c.stream>>>(sc, w, n, o, d, uv, src, first, tmax, any_hit);
}
void mfx_f_seam_read(const LaunchCfg &c, const SceneF &sc, const WaveF &w, int n, long long first, int any_hit, int *prim, int *sub, double *t)
{
    k_f_seam_read<<<persistent_blocks(k_f_seam_read, 256, c.blocks), 256, 0, c.stream>>>(sc, w, n, first, any_hit, prim, sub, t);
}
void mfx_accum_ray_totals(cudaStream_t s, const int *counts, int ext_lo, int ext_n, int sh_lo, int sh_n, unsigned long long *totals)
{
    k_accum_totals<<<1, 1, 0, s>>>(counts, ext_lo, ext_n, sh_lo, sh_n, totals);
}
void mfx_film_add(cudaStream_t s, TileMap tm, int width, double *sum, const double *frame, double *target, double fc)
{
    k_film_add<<<592, 256, 0, s>>>(tm, width, sum, frame, target, fc);
}
void mfx_film_tonemap(cudaStream_t s, TileMap tm, int width, const double *target_wh, uint8_t *rgba8)
{
    k_film_tonemap<<<592, 256, 0, s>>>(tm, width, target_wh, rgba8);
}
void mfx_film_display_sky(cudaStream_t s, TileMap tm, int width, const double *target_wh, uint8_t *rgba8)
{
    k_film_display_sky<<<592, 256, 0, s>>>(tm, width, target_wh, rgba8);
}
