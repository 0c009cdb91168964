// mfx_hybrid.cu -- id-exact closest hits at wavefront speed.  COMPILED WITH --fmad=false.
//
// north_star: "primary-hit buffers (triangle/sphere ID) must be bit-exact".  The reference's closest-hit query
// (Bvh.CheckHit, BvhNode.fs:62-83) has one deterministic answer:
//     the smallest t over every primitive the exhaustive walk tests;
//     equal t: the leaf later in depth-first order wins (`if l.t < r.t then l else r`, :69-70), inside a leaf the
//     first minimal key (`Array.minBy`, :76-80);
//     a primitive is tested iff AABB.hit (IHitable.fs:18-54) passes for its leaf and every ancestor.
// That answer does not depend on the tree that finds it, so this kernel walks the library's own SAH tree with the
// persistent-warp machinery of k_f_trace6 (mfx_fast.cu) and makes only the DECISIONS in f64:
//   * node step: f32 slab tests, boxes padded per ray by 4e-6 x (|scene| + |origin|) -- eight times the worst
//     accumulated rounding between the f64 ray and the f32 arithmetic (ray rounded to f32, rcp.approx, o/d product,
//     fma) -- so a box that holds an f64 hit is never culled; the t-shrink limit is best_t rounded UP to f32 and a
//     node is culled only when its (padded, rounded-down) entry lies strictly beyond it: exact ties survive;
//   * leaf: every candidate primitive runs the exact kernel's arithmetic (Triangle.Hit as tri_eval_x = tri_hit_x without
//     early exits, sphere_hit_x / sphere_hit_sky_x of mfx_exact_dev.cuh) on f64 records laid out in the own tree's
//     slot order (PrimH: the very edge vectors of the exact layout), with the f64 ray -- the same operations, the same t;
//   * ties: resolved with the reference tree's leaf table (leaf_of_ref), tree-independent;
//   * the winner's reference leaf box is re-tested with AABB.hit verbatim.  Child boxes nest exactly (Bound.Union is
//     min/max) and every operation of the slab test is monotone in the box, so a leaf box that passes implies all
//     its ancestors pass: one test decides "the reference reaches this primitive".  A winner that fails it, a
//     direction with a zero component (0/0 breaks the monotonicity argument) or a hit at t >= tMax (quirk Q2: the
//     tMax-blind triangle) is handed to the exact kernel's traversal in k_h_fixup -- measure-zero cases, but the
//     answer never depends on luck.
// MFX_SKY_TRACER: ListHit (RayTracing.fs:256-258) tests every sphere, ties go to the smaller list index; no box
// check, no fixup.
#include "mfx_exact_dev.cuh"
#include "mfx_fast_dev.cuh"
#include <algorithm>

#define HYB_REF_MASK 0x3fffffff
#define HYB_TMIN_BOX 1e-30f          // keys must stay positive floats (integer order == float order)

struct HybBest { double t; int ref; };

// exact tie rule between two hits of equal t (see the header); a, b = exact slots
__device__ __forceinline__ bool hyb_tie_wins(const int *leaf_of_ref, const int *ref_id, int sky, int a, int b)
{
    if (sky) return ref_id[a] < ref_id[b];                  // ListHit keeps the first minimal t in list order
    const int la = leaf_of_ref[a], lb = leaf_of_ref[b];
    return (la == lb) ? (a < b) : (a > b);                  // leaves partition the slot range in depth-first order
}

// Triangle.PreCalcu + Hit (Trangle.fs:120-155) with the SAME operations as tri_hit_x but no early exits: every value is
// computed, the acceptance rules are evaluated afterwards in the reference's order.  Identical results (a rejected
// triangle's later values are simply never looked at), and two of these inline into independent dependency chains.
__device__ __forceinline__ bool tri_eval_x(D3 v0, D3 e1, D3 e2, D3 o, D3 dir, double tMin, double &t)
{
    const D3 s1 = cross(dir, e2);
    const double divisor = dot(s1, e1);
    const double inv = 1. / divisor;
    const D3 d = o - v0;
    const double b1 = dot(d, s1) * inv;
    const D3 s2 = cross(d, e1);
    const double b2 = dot(dir, s2) * inv;
    t = dot(e2, s2) * inv;
    return !(fabs(divisor) < 1e-6) && !(b1 < 0. || b1 > 1.) && !(b2 < 0. || (b1 + b2) >= 1.) && (t > tMin);
}

// IHitable.Hit on one own-tree slot record.  kind 0: a Triangle, or the first triangle of a Rect (Rect.Hit returns it
// whenever it hits, Rect.fs:27-29); kind 1: the second triangle of a Rect -- Rect.Hit answers with it only if the first
// one misses (:30-31, quirk Q3), so both are tested; kind 2: Sphere.
__device__ __forceinline__ bool slot_eval_x(const PrimH *p, int kind, D3 v0, D3 e1, D3 e2, D3 o, D3 d, double tMin, double tMax, int sky, double &t, int &sub)
{
    sub = 0;
    if (kind == 2) return sky ? sphere_hit_sky_x(v0, e1.x, o, d, tMin, tMax, t) : sphere_hit_x(v0, e1.x, o, d, tMin, tMax, t);
    bool hit = tri_eval_x(v0, e1, e2, o, d, tMin, t);
    if (kind == 1 && !hit) { sub = 1; hit = tri_eval_x(v0, e2, ld3(p->e3), o, d, tMin, t); }
    return hit;
}

// Tests the slots of one own-tree leaf in f64.  Out of line: its f64 registers must not cost the traversal loop its
// occupancy (the loop itself holds no f64 state but best.t).  HYB_LEAF_PAIRED (A/B knob): two slots at a time without
// early exits -- measured slower (C2 primary rays 10.9 against 12.3 Grays/s): the phase is bound by f64 issue, not by
// f64 latency, so the early exits of tri_hit_x pay.
__device__ __noinline__ HybBest hyb_leaf(const PrimH *ph, const int *leaf_of_ref, const int *ref_id,
                                         D3 o, const double *dir, int meta, double tMin, double tMax, int sky, HybBest best)
{
    const D3 d = mk3<double>(dir[0], dir[1], dir[2]);
    const int first = meta >> 3, cnt = meta & 7;
#ifdef HYB_LEAF_PAIRED
    for (int k = 0; k < cnt; k += 2) {
        const PrimH *pa = ph + first + k, *pb = (k + 1 < cnt) ? pa + 1 : pa;
        const D3 av0 = ld3(pa->v0), ae1 = ld3(pa->e1), ae2 = ld3(pa->e2);
        const D3 bv0 = ld3(pb->v0), be1 = ld3(pb->e1), be2 = ld3(pb->e2);
        const int akind = pa->kind, aref = pa->ref, bkind = pb->kind, bref = pb->ref;
        double ta, tb; int suba, subb;
        const bool hita = slot_eval_x(pa, akind, av0, ae1, ae2, o, d, tMin, tMax, sky, ta, suba);
        const bool hitb = slot_eval_x(pb, bkind, bv0, be1, be2, o, d, tMin, tMax, sky, tb, subb) && (k + 1 < cnt);
        if (hita && aref != (best.ref & HYB_REF_MASK) &&
            (best.ref < 0 || ta < best.t || (ta == best.t && hyb_tie_wins(leaf_of_ref, ref_id, sky, aref, best.ref & HYB_REF_MASK)))) {
            best.t = ta; best.ref = aref | (suba << 30);
        }
        if (hitb && bref != (best.ref & HYB_REF_MASK) &&
            (best.ref < 0 || tb < best.t || (tb == best.t && hyb_tie_wins(leaf_of_ref, ref_id, sky, bref, best.ref & HYB_REF_MASK)))) {
            best.t = tb; best.ref = bref | (subb << 30);
        }
    }
#else
    for (int k = 0; k < cnt; k++) {
        const PrimH *p = ph + first + k;
        const int kind = p->kind, ref = p->ref;
        if (ref == (best.ref & HYB_REF_MASK)) continue;             // the other half of the Rect that leads already
        const D3 v0 = ld3(p->v0);
        double t; int sub = 0; bool hit;
        if (kind == 2) hit = sky ? sphere_hit_sky_x(v0, p->e1[0], o, d, tMin, tMax, t) : sphere_hit_x(v0, p->e1[0], o, d, tMin, tMax, t);
        else {
            const D3 e1 = ld3(p->e1), e2 = ld3(p->e2);
            hit = tri_hit_x(v0, e1, e2, o, d, tMin, t);
            if (kind == 1 && !hit) { sub = 1; hit = tri_hit_x(v0, e2, ld3(p->e3), o, d, tMin, t); }   // Rect.Hit: tri1 else tri2 (Rect.fs:26-31)
        }
        if (!hit) continue;
        if (best.ref < 0 || t < best.t || (t == best.t && hyb_tie_wins(leaf_of_ref, ref_id, sky, ref, best.ref & HYB_REF_MASK))) {
            best.t = t; best.ref = ref | (sub << 30);
        }
    }
#endif
    return best;
}

// Does the reference's walk reach the winner?  AABB.hit on its leaf box (see the header) -- decided WITHOUT the six
// divisions whenever the hit point p = o + t d sits robustly inside the box: then on every axis the slab's entry parameter
// is below t and its exit parameter above t by far more than the rounding of `(plane - o) / d` (2^-53 relative; the
// margin here is 1e-10 of the summed magnitudes involved), so every comparison AABB.hit makes between an entry and an exit of
// two DIFFERENT axes (IHitable.fs:38-52 never compares an axis with itself) comes out "overlap", and tmin < tMax,
// tmax > tMin follow from tMin < t < tMax.  One axis may be flat (an axis-aligned quad's box has no thickness: entry and
// exit are then the SAME expression, both within rounding of t).  Anything less clear-cut -- the point within the margin
// of a face, two flat axes, t within the margin of tMin -- runs AABB.hit verbatim.
__device__ __noinline__ bool hyb_verify(const NodeX *nodes, const int *leaf_of_ref, D3 o, const double *dir, int ref, double tMin, double tMax, double t)
{
    const D3 d = mk3<double>(dir[0], dir[1], dir[2]);
    if (d.x == 0. || d.y == 0. || d.z == 0.) return false;
    if (!(t < tMax)) return false;
    const NodeX *nd = nodes + leaf_of_ref[ref & HYB_REF_MASK];
    const double lo[3] = { nd->pmin[0], nd->pmin[1], nd->pmin[2] }, hi[3] = { nd->pmax[0], nd->pmax[1], nd->pmax[2] };
    const double oo[3] = { o.x, o.y, o.z }, dd[3] = { d.x, d.y, d.z };
    // S bounds every magnitude that enters the slab expressions; inside-margin 1e-10 S in space is >= 1e-10 S in t (|d| <= 1),
    // a flat axis is pinned to 1e-13 S in space and needs |d_a| >= 1e-3, i.e. to 1e-10 S in t: below every other margin
    double S = fabs(t) + fabs(tMin);
#pragma unroll
    for (int a = 0; a < 3; a++) S += fabs(oo[a]) + fabs(lo[a]) + fabs(hi[a]);
    const double m_in = 1e-10 * S, m_flat = 1e-13 * S;
    int flat = 0; bool clear = (t > tMin + m_in) && (t < tMax - 1e-10 * fabs(tMax));
#pragma unroll
    for (int a = 0; a < 3; a++) {
        const double p = oo[a] + t * dd[a];
        const bool inside = (p >= lo[a] + m_in) && (p <= hi[a] - m_in);
        const bool on_flat = (hi[a] == lo[a]) && (fabs(p - lo[a]) <= m_flat) && (fabs(dd[a]) >= 1e-3);
        flat += on_flat ? 1 : 0;
        clear = clear && (inside || on_flat);
    }
    if (clear && flat <= 1) return true;
    double e;
    return aabb_hit_x(*nd, o, d, tMin, tMax, e);
}

// the ray origin: one constant for a pinhole frame (the camera), per ray otherwise
__device__ __forceinline__ D3 hyb_origin(const WaveH &wh, const D3 &cam_o, int cam0, int pid)
{
    if (cam0) return cam_o;
    const double *p = wh.org64 + 3 * (size_t)pid;
    return mk3<double>(p[0], p[1], p[2]);
}

// seam != 0 (Bvh.Hit / GetRay + Hit seams): the exact slot and the f64 t are kept; frames only need w.hit.
template <int REFILL_T, int LEAF_T, int NSTEP, int MINB>
__global__ void __launch_bounds__(FAST_BLOCK, MINB) k_h_trace(SceneF sc, const NodeX *nodes, const int *ref_id,
                                                              SceneH sh, WaveF w, WaveH wh, int bounce, HybQuery q, D3 cam_o, int cam0, int seam)
{
    extern __shared__ uint2 s_stack[];              // [stack_smem][FAST_BLOCK]
    uint2 *my_stack = s_stack + threadIdx.x;
    const int S = sc.stack_smem;
    uint2 *my_spill = sc.stack_spill + ((size_t)blockIdx.x * FAST_BLOCK + threadIdx.x);
    const size_t spill_stride = (size_t)sc.spill_threads;
    const unsigned FULL = 0xffffffffu;
    const unsigned lane = threadIdx.x & 31u;
    const int n = w.counts[bounce];
    int *cursor = &w.counts[CUR_EXT(bounce)];

    int pid = -1;
    F3 idir = f3(0.f, 0.f, 0.f), ood_n = idir, ood_f = idir;
    float limit = 0.f;
    HybBest best; best.t = 0.; best.ref = -1;
    int node = 0, sp = 0;
    bool needPop = false;
    int leafA = -1;
    bool exhausted = false;
    unsigned iters = 0u;

    for (;;) {
        const unsigned idle = __ballot_sync(FULL, pid < 0);
        unsigned idle_now = idle;
        if (++iters > (1u << 22)) { if (lane == 0) atomicAdd(&w.counts[MFX_COUNTS_LEN - 1], 1); break; }   // watchdog
        if (!exhausted && __popc(idle) >= REFILL_T) {
            const int nidle = __popc(idle);
            int base = 0;
            if (lane == 0) base = atomicAdd(cursor, nidle);
            base = __shfl_sync(FULL, base, 0);
            if (base + nidle >= n) exhausted = true;
            if (pid < 0) {
                const int idx = base + __popc(idle & ((1u << lane) - 1u));
                if (idx < n) {
                    pid = idx;
                    const double *dir = wh.dir64 + 3 * (size_t)pid;
                    const D3 o64 = hyb_origin(wh, cam_o, cam0, pid);
                    const F3 o = f3((float)o64.x, (float)o64.y, (float)o64.z);
                    const F3 d = f3((float)dir[0], (float)dir[1], (float)dir[2]);
                    const RayF r = make_ray_fast(o, d, HYB_TMIN_BOX, -1);
                    idir = r.idir;
                    // per-ray pad: every box plane moves outward by `pad` in space = pad * |1/d| in t
                    const float pad = sh.pad_factor * (sh.max_abs + fmaxf(fabsf(o.x), fmaxf(fabsf(o.y), fabsf(o.z))));
                    const F3 pt = f3(pad * fabsf(idir.x), pad * fabsf(idir.y), pad * fabsf(idir.z));
                    ood_n = r.ood + pt; ood_f = r.ood - pt;
                    limit = 3.0e38f;                         // triangles ignore tMax (Trangle.fs:148): nothing is culled by it
                    best.t = 0.; best.ref = -1; sp = 0; leafA = -1; node = 0; needPop = false;
                }
            }
            idle_now = __ballot_sync(FULL, pid < 0);
        }
        if (idle_now == FULL) { if (exhausted) break; continue; }

        const bool px = idir.x >= 0.f, py = idir.y >= 0.f, pz = idir.z >= 0.f;
#pragma unroll
        for (int rep = 0; rep < NSTEP; rep++)
        if (pid >= 0 && leafA < 0 && !needPop) {
            const QuadF *qp = sc.quads + node;
            float4 lox, hix, loy, hiy, loz, hiz, m4, pad4;
            ldg8(&qp->lox, lox, hix); ldg8(&qp->loy, loy, hiy); ldg8(&qp->loz, loz, hiz); ldg8(&qp->meta, m4, pad4);
            unsigned key[4];
#define QUAD_SLOT(S_, C)                                                                                             \
            {                                                                                                        \
                const float nx = fmaf(px ? lox.C : hix.C, idir.x, -ood_n.x), fx = fmaf(px ? hix.C : lox.C, idir.x, -ood_f.x); \
                const float ny = fmaf(py ? loy.C : hiy.C, idir.y, -ood_n.y), fy = fmaf(py ? hiy.C : loy.C, idir.y, -ood_f.y); \
                const float nz = fmaf(pz ? loz.C : hiz.C, idir.z, -ood_n.z), fz = fmaf(pz ? hiz.C : loz.C, idir.z, -ood_f.z); \
                const float tn = fmaxf(fmaxf(nx, ny), fmaxf(nz, HYB_TMIN_BOX));                                      \
                const float tf = fminf(fminf(fx, fy), fminf(fz, limit));                                             \
                const int mt = __float_as_int(m4.C);                                                                 \
                key[S_] = (tn <= tf && mt != MFX_QUAD_EMPTY) ? ((__float_as_uint(tn) & ~7u) | (mt >= 0 ? 4u : 0u) | (unsigned)S_) : KEY_INF; \
            }
            QUAD_SLOT(0, x) QUAD_SLOT(1, y) QUAD_SLOT(2, z) QUAD_SLOT(3, w)
#undef QUAD_SLOT
            // sorting network (0,1)(2,3)(0,2)(1,3)(1,2)
            unsigned a0 = umin_(key[0], key[1]), a1 = umax_(key[0], key[1]);
            unsigned a2 = umin_(key[2], key[3]), a3 = umax_(key[2], key[3]);
            const unsigned k0 = umin_(a0, a2), t2 = umax_(a0, a2);
            const unsigned t1 = umin_(a1, a3), k3 = umax_(a1, a3);
            const unsigned k1 = umin_(t1, t2), k2 = umax_(t1, t2);
            const bool any0 = k0 != KEY_INF;
            const bool leaf0 = any0 && (k0 & 4u);
            const int c0 = pick4(m4, k0 & 3u);
            leafA = leaf0 ? c0 : -1;
            const int m = (k1 != KEY_INF ? 1 : 0) + (k2 != KEY_INF ? 1 : 0) + (k3 != KEY_INF ? 1 : 0);
#define STACK_PUT(I, K)                                                                                              \
            { const int i_ = (I); const uint2 v_ = make_uint2((K), (unsigned)node);                                  \
              DBG_CHECK(i_ >= 0 && i_ < 3 * sc.own_depth, w.counts);                                                  \
              DBG_CHECK(i_ < S || blockIdx.x * FAST_BLOCK + threadIdx.x < (unsigned)sc.spill_threads, w.counts);       \
              if (i_ < S) my_stack[(size_t)i_ * FAST_BLOCK] = v_; else my_spill[(size_t)(i_ - S) * spill_stride] = v_; }
            if (m >= 1) STACK_PUT(sp + m - 1, k1)
            if (m >= 2) STACK_PUT(sp + m - 2, k2)
            if (m >= 3) STACK_PUT(sp, k3)
#undef STACK_PUT
            sp += m;
            const bool descend = any0 && !leaf0;
            needPop = !descend;
            if (descend) node = ~c0;
            DBG_CHECK(!descend || (unsigned)node < (unsigned)sc.n_quads, w.counts);
            DBG_CHECK(leafA < 0 || ((leafA >> 3) >= 0 && (leafA >> 3) + (leafA & 7) <= sc.n_slots), w.counts);
        }
        bool finished = false;
        const unsigned lp = __ballot_sync(FULL, pid >= 0 && leafA >= 0);
        if (lp) {
            const unsigned nd = ~idle_now & ~lp;
            if (__popc(lp) >= LEAF_T || nd == 0u) {
                if (pid >= 0 && leafA >= 0) {
                    best = hyb_leaf(sh.prims_h, sh.leaf_of_ref, ref_id, hyb_origin(wh, cam_o, cam0, pid), wh.dir64 + 3 * (size_t)pid,
                                    leafA, q.tmin, q.tmax, q.sky, best);
                    if (best.ref >= 0) limit = __double2float_ru(best.t);
                    leafA = -1;
                }
            }
        }
        if (pid >= 0 && needPop && leafA < 0) {
            for (;;) {
                if (sp == 0) { finished = true; break; }
                --sp;
                const uint2 e = (sp < S) ? my_stack[(size_t)sp * FAST_BLOCK] : my_spill[(size_t)(sp - S) * spill_stride];
                if (__uint_as_float(e.x & ~7u) <= limit) {
                    const int link = __ldg(reinterpret_cast<const int *>(&sc.quads[e.y].meta) + (e.x & 3u));
                    if (e.x & 4u) leafA = link;
                    else { node = ~link; needPop = false; }
                    break;
                }
            }
        }
        if (finished) {
            int ref = best.ref;
            if (ref >= 0 && !q.sky && !hyb_verify(nodes, sh.leaf_of_ref, hyb_origin(wh, cam_o, cam0, pid), wh.dir64 + 3 * (size_t)pid, ref, q.tmin, q.tmax, best.t)) ref = -2;
            if (ref == -2) {
                const int at = atomicAdd(wh.fix_n, 1);
                if (at < MFX_HYB_FIX_CAP) wh.fix_q[at] = pid;
            }
            DBG_CHECK(pid >= 0 && pid < w.P && (ref < 0 || (ref & HYB_REF_MASK) < sh.n_ref), w.counts);
            if (seam) { wh.ref[pid] = ref; wh.t[pid] = best.t; }
            int fs = ref;                                   // -1 miss, -2 waiting for k_h_fixup
            if (ref >= 0) { const int2 f = __ldg(sh.ref_fslot + (ref & HYB_REF_MASK)); fs = (ref >> 30) ? f.y : f.x; }
            w.hit[pid] = make_float2((float)best.t, __int_as_float(fs));
            pid = -1;
        }
    }
}

// The rays k_h_trace could not clear (see the header) take the exact kernel's walk of the reference tree.
__global__ void __launch_bounds__(128) k_h_fixup(SceneX sx, SceneH sh, WaveF w, WaveH wh, int bounce, HybQuery q, int cam0, int seam)
{
    const int flagged = *wh.fix_n;
    if (flagged == 0) return;
    const bool scan = flagged > MFX_HYB_FIX_CAP;
    const int n = scan ? w.counts[bounce] : flagged;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int pid = scan ? i : wh.fix_q[i];
        if (__float_as_int(w.hit[pid].y) != -2) continue;
        const double *dir = wh.dir64 + 3 * (size_t)pid;
        const D3 o = hyb_origin(wh, ld3(sx.cam.pos), cam0, pid), d = mk3<double>(dir[0], dir[1], dir[2]);
        const HitX h = q.sky ? sky_hit_x<false>(sx, o, d, q.tmin, q.tmax, nullptr) : bvh_hit_x<false, false>(sx, o, d, q.tmin, q.tmax, nullptr);
        const int ref = (h.slot < 0) ? -1 : (h.slot | (h.sub << 30));
        if (seam) { wh.ref[pid] = ref; wh.t[pid] = h.t; }
        int fs = -1;
        if (ref >= 0) { const int2 f = sh.ref_fslot[h.slot]; fs = h.sub ? f.y : f.x; }
        w.hit[pid] = make_float2((float)h.t, __int_as_float(fs));
    }
}

// Ray generation of a wave whose bounce 0 is traced id-exactly: PixelIntegrator.Sample's jitter and cam.GetRay
// (Integrators.fs:166-169, Camera.fs:134-139; RayTraceCamera.GetRay for the sphere sample) in f64 with the reference's
// operation order -- the very rays the exact mode generates -- kept in f64 for k_h_trace and rounded once for the
// f32 shading that follows.
__global__ void __launch_bounds__(256) k_h_raygen(SceneF sc, SceneX sx, WaveF w, WaveH wh, TileMap tm, int pix0, int npix, int s0, int S, uint64_t seed)
{
    const long long total = (long long)npix * S;
    for (long long pid = (long long)blockIdx.x * blockDim.x + threadIdx.x; pid < total; pid += (long long)gridDim.x * blockDim.x) {
        int sl, pl;
        path_split(tm, pid, npix, sl, pl);
        int pix, px, py;
        pixel_of(tm, sx.width, pix0 + pl, pix, px, py);
        RngX g; g.pixel = (uint32_t)pix; g.sample = (uint32_t)(s0 + sl); g.k0 = (uint32_t)seed; g.k1 = (uint32_t)(seed >> 32);
        double u4[4];
        rng_draw_x(g, MFX_DIM_CAMERA, 0, u4);
        const double u = ((double)px + u4[0]) / (double)sx.width;
        const double v = ((double)py + u4[1]) / (double)sx.height;
        D3 d, org = ld3(sx.cam.pos);
        if (sx.mode == MFX_MODE_SKY) lens_ray_x(sx.cam, sx.lens, u, v, sx.lens.radius != 0.0 ? &g : nullptr, org, d);
        else d = camera_ray_dir_x(sx.cam, u, v);
        double *dir = wh.dir64 + 3 * (size_t)pid;
        dir[0] = d.x; dir[1] = d.y; dir[2] = d.z;
        if (!w.cam_origin) {
            double *op = wh.org64 + 3 * (size_t)pid;
            op[0] = org.x; op[1] = org.y; op[2] = org.z;
            w.ray_o[0][pid] = make_float4((float)org.x, (float)org.y, (float)org.z, __int_as_float(-1));
        }
        w.ray_d[0][pid] = make_float4((float)d.x, (float)d.y, (float)d.z, __int_as_float((int)pid));
        w.rad[pid] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (pid == 0) w.counts[0] = (int)total;
    }
}

// Finer seams (Bvh.Hit, GetRay + Hit) through the hybrid kernel: the f64 rays go into the wave's ray64 queue.
__global__ void __launch_bounds__(256) k_h_seam_setup(SceneX sx, WaveF w, WaveH wh, int n, const double *o, const double *d, const double *uv, long long first)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const long long r = first + i;
        D3 oo, dd;
        if (d) {
            oo = mk3<double>(o[3 * r], o[3 * r + 1], o[3 * r + 2]);
            dd = mk3<double>(d[3 * r], d[3 * r + 1], d[3 * r + 2]);
            if (sx.mode == MFX_MODE_SKY) dd = normalize_x(dd);          // Ray(origin, direc) normalises (RayTracing.fs:14-16)
        } else {
            double u, v;
            if (uv) { u = uv[2 * r]; v = uv[2 * r + 1]; }
            else {
                const int j = (int)(r / sx.width), ii = (int)(r - (long long)j * sx.width);
                u = ((double)ii + 0.5) / (double)sx.width;
                v = ((double)j + 0.5) / (double)sx.height;
            }
            if (sx.mode == MFX_MODE_SKY) lens_ray_x(sx.cam, sx.lens, u, v, nullptr, oo, dd);
            else { oo = ld3(sx.cam.pos); dd = camera_ray_dir_x(sx.cam, u, v); }
        }
        double *op = wh.org64 + 3 * (size_t)i, *dp = wh.dir64 + 3 * (size_t)i;
        op[0] = oo.x; op[1] = oo.y; op[2] = oo.z; dp[0] = dd.x; dp[1] = dd.y; dp[2] = dd.z;
        if (i == 0) w.counts[0] = n;
    }
}

__global__ void __launch_bounds__(256) k_h_seam_read(SceneX sx, WaveH wh, int n, long long first, int *prim, int *sub, double *t)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const long long r = first + i;
        const int ref = wh.ref[i];
        if (ref < 0) { prim[r] = -1; if (sub) sub[r] = 0; t[r] = 0.; }
        else { prim[r] = sx.ref_id[ref & HYB_REF_MASK]; if (sub) sub[r] = ref >> 30; t[r] = wh.t[i]; }
    }
}

// MFX_EXACT_F64 frames through the same kernel: the closest-hit queries of the exact wavefront (WaveX: f64 SoA by path id,
// queues of path ids) are gathered into the hybrid's queue, traced, and scattered back.  bvh_hit_x and k_h_trace return
// the same (slot, sub, t) by construction, so the frames stay bit-identical -- at a fraction of the f64 box tests.
__global__ void __launch_bounds__(256) k_h_gather_x(WaveX wx, WaveF w, WaveH wh, int bounce)
{
    const int n = wx.counts[bounce];
    const int *q = wx.queue[bounce & 1];
    const size_t P = (size_t)wx.P;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int pid = q[i];
        double *op = wh.org64 + 3 * (size_t)i, *dp = wh.dir64 + 3 * (size_t)i;
        op[0] = wx.ray_o[pid]; op[1] = wx.ray_o[P + pid]; op[2] = wx.ray_o[2 * P + pid];
        dp[0] = wx.ray_d[pid]; dp[1] = wx.ray_d[P + pid]; dp[2] = wx.ray_d[2 * P + pid];
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) { w.counts[0] = n; w.counts[CUR_EXT(0)] = 0; }
}

__global__ void __launch_bounds__(256) k_h_scatter_x(WaveX wx, WaveH wh, int bounce)
{
    const int n = wx.counts[bounce];
    const int *q = wx.queue[bounce & 1];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int pid = q[i];
        const int ref = wh.ref[i];
        wx.hit_t[pid] = wh.t[i];
        wx.hit_slot[pid] = ref;                     // -1 miss, else exact slot | sub << 30: WaveX's own convention
    }
}

// ---------------------------------------------------------------- exact shadow queries without ~46 f64 box tests per ray
// SingleDirectLightIntegrator.Eval asks `bvh.Hit(shadowRay, 1e-6, dist - 1e-6).hit` (Integrators.fs:44).  CheckHit's answer
// is "some leaf the walk reaches yields a hit record": a leaf is reached iff AABB.hit passes for it and its ancestors -- and,
// boxes nesting exactly and the slab test being monotone in the box, iff it passes for the LEAF's own box (fixed tMin, tMax);
// its record is Array.minBy (hit ? t : tMax) over its <= 3 primitives (BvhNode.fs:76-80: tMax-blind triangles, quirk Q2,
// included).  So the walk over the interior nodes only has to VISIT A SUPERSET of the reachable leaves: it runs on the f32
// copy of the reference tree (PairF: both children of a heap node in 64 bytes, boxes rounded outward) with the per-ray pad
// of k_h_trace, and every visited leaf is then decided exactly -- AABB.hit verbatim on its f64 box, prim_hit_x on its
// primitives in index order.  Two f64 box tests per ray instead of forty-six.  A direction with a zero component (the
// 0/0 family of AABB.hit, where monotonicity fails) or a window that ends at or before the origin (a light sample closer
// than 1e-6: the f32 test clips the near side at 0) takes bvh_hit_x.
__device__ __noinline__ bool shadow_leaf_x(const NodeX *nodes, const PrimX *prims, int node0, D3 o, D3 d, double tMin, double tMax)
{
    const NodeX nd = nodes[node0];
    double e;
    if (!aabb_hit_x(nd, o, d, tMin, tMax, e)) return false;             // the reference's walk does not reach this leaf
    bool have = false, recHit = false; double bestKey = 0.;
    for (int k = 0; k < nd.count; k++) {
        const PrimX p = prims[nd.first + k];
        double t; int sub;
        const bool h = prim_hit_x(p, o, d, tMin, tMax, t, sub);
        const double key = h ? t : tMax;
        if (!have || key < bestKey) { have = true; bestKey = key; recHit = h; }
    }
    return recHit;
}

__global__ void __launch_bounds__(128) k_h_shadow_x(SceneX sx, const PairF *pairs, float3 root_lo, float3 root_hi, int root_meta,
                                                    WaveX w, int bounce, float max_abs, float pad_factor)
{
    const int n = w.counts[bounce + 1];                 // the paths shaded at vertex `bounce` (k_x_shadow's convention)
    const int *q = w.queue[(bounce + 1) & 1];
    const size_t P = (size_t)w.P;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int pid = q[i];
        const D3 o = mk3<double>(w.ray_o[pid], w.ray_o[P + pid], w.ray_o[2 * P + pid]);   // hit.point
        const D3 d = mk3<double>(w.sh_d[pid], w.sh_d[P + pid], w.sh_d[2 * P + pid]);
        const double tMin = 1e-6, tMax = w.sh_dist[pid] - 1e-6;
        bool occluded;
        if (d.x == 0. || d.y == 0. || d.z == 0. || !(tMax > 0.)) occluded = bvh_hit_x<true, false>(sx, o, d, tMin, tMax, nullptr).slot >= 0;
        else {
            occluded = false;
            const F3 of = f3((float)o.x, (float)o.y, (float)o.z), df = f3((float)d.x, (float)d.y, (float)d.z);
            const RayF r = make_ray_fast(of, df, HYB_TMIN_BOX, -1);
            const float pad = pad_factor * (max_abs + fmaxf(fabsf(of.x), fmaxf(fabsf(of.y), fabsf(of.z))));
            const F3 pt = f3(pad * fabsf(r.idir.x), pad * fabsf(r.idir.y), pad * fabsf(r.idir.z));
            const F3 on = r.ood + pt, ofar = r.ood - pt;
            const bool px = r.idir.x >= 0.f, py = r.idir.y >= 0.f, pz = r.idir.z >= 0.f;
            const float lim = __double2float_ru(tMax) * 1.000001f + 1e-30f;
#define HS_BOX(lx, ly, lz, hx, hy, hz)                                                                                  \
            (fmaxf(fmaxf(fmaf(px ? (lx) : (hx), r.idir.x, -on.x), fmaf(py ? (ly) : (hy), r.idir.y, -on.y)),                 \
                   fmaxf(fmaf(pz ? (lz) : (hz), r.idir.z, -on.z), 0.f)) <=                                                  \
             fminf(fminf(fmaf(px ? (hx) : (lx), r.idir.x, -ofar.x), fmaf(py ? (hy) : (ly), r.idir.y, -ofar.y)),             \
                   fminf(fmaf(pz ? (hz) : (lz), r.idir.z, -ofar.z), lim)))
            if (HS_BOX(root_lo.x, root_lo.y, root_lo.z, root_hi.x, root_hi.y, root_hi.z)) {
                if (root_meta >= 0) occluded = shadow_leaf_x(sx.nodes, sx.prims, 0, o, d, tMin, tMax);
                else {
                    unsigned stack[40];
                    int sp = 0;
                    unsigned h = 1u;                                    // 1-based heap index of the interior node to expand
                    for (int guard = 0; guard < (1 << 24); guard++) {
                        const PairF *pp = pairs + h;
                        const float4 q0 = ldg4(&pp->q0), q1 = ldg4(&pp->q1), q2 = ldg4(&pp->q2), q3 = ldg4(&pp->q3);
                        const bool hitL = HS_BOX(q0.x, q0.y, q0.z, q0.w, q1.x, q1.y), hitR = HS_BOX(q1.z, q1.w, q2.x, q2.y, q2.z, q2.w);
                        const bool leafL = __float_as_int(q3.x) >= 0, leafR = __float_as_int(q3.y) >= 0;
                        if (hitL && leafL && shadow_leaf_x(sx.nodes, sx.prims, (int)(2u * h) - 1, o, d, tMin, tMax)) { occluded = true; break; }
                        if (hitR && leafR && shadow_leaf_x(sx.nodes, sx.prims, (int)(2u * h), o, d, tMin, tMax)) { occluded = true; break; }
                        const bool inL = hitL && !leafL, inR = hitR && !leafR;
                        if (inL && inR) { if (sp < 40) stack[sp++] = 2u * h + 1u; h = 2u * h; }
                        else if (inL) h = 2u * h;
                        else if (inR) h = 2u * h + 1u;
                        else if (sp > 0) h = stack[--sp];
                        else break;
                    }
                }
            }
#undef HS_BOX
        }
        if (occluded) {
            const size_t vb = (size_t)bounce * 3 * P;
            w.v_l[vb + pid] = 0.; w.v_l[vb + P + pid] = 0.; w.v_l[vb + 2 * P + pid] = 0.;
        }
    }
}

// the exact wavefront keeps its own counts: the hybrid kernel's watchdog / debug-check flags live in WaveF.counts
__global__ void k_h_guard(int *counts, unsigned long long *totals)
{
    totals[3] += (unsigned)counts[MFX_COUNTS_LEN - 1]; totals[5] += (unsigned)counts[MFX_DBG_SLOT];
    counts[MFX_COUNTS_LEN - 1] = 0; counts[MFX_DBG_SLOT] = 0;
}

__global__ void k_h_accum(const int *fix_n, unsigned long long *total) { *total += (unsigned)*fix_n; }

// ---------------------------------------------------------------- launchers
void mfx_h_accum_fixups(cudaStream_t s, const WaveH &wh, unsigned long long *total) { k_h_accum<<<1, 1, 0, s>>>(wh.fix_n, total); }
void mfx_h_raygen(const LaunchCfg &c, const SceneF &sc, const SceneX &sx, const WaveF &w, const WaveH &wh, TileMap tm, int pix0, int npix,
                  int s0, int S, uint64_t seed)
{
    k_h_raygen<<<persistent_blocks(k_h_raygen, 256, c.blocks), 256, 0, c.stream>>>(sc, sx, w, wh, tm, pix0, npix, s0, S, seed);
}
void mfx_h_seam_setup(const LaunchCfg &c, const SceneX &sx, const WaveF &w, const WaveH &wh, int n, const double *o, const double *d,
                      const double *uv, long long first)
{
    k_h_seam_setup<<<persistent_blocks(k_h_seam_setup, 256, c.blocks), 256, 0, c.stream>>>(sx, w, wh, n, o, d, uv, first);
}
template <int RT, int LT, int NS, int MB>
static void launch_h_trace(const LaunchCfg &c, const SceneF &sc, const SceneX &sx, const SceneH &sh, const WaveF &w, const WaveH &wh, int bounce, HybQuery q, int seam)
{
    const size_t smem = (size_t)sc.stack_smem * FAST_BLOCK * sizeof(uint2);
    auto kern = k_h_trace<RT, LT, NS, MB>;
    int blocks = persistent_blocks(kern, FAST_BLOCK, c.blocks, smem);
    if (sc.stack_spill && blocks * FAST_BLOCK > sc.spill_threads) blocks = sc.spill_threads / FAST_BLOCK;
    if (c.max_items > 0) blocks = std::max(1, std::min(blocks, (c.max_items + FAST_BLOCK - 1) / FAST_BLOCK));
    D3 cam_o; cam_o.x = sx.cam.pos[0]; cam_o.y = sx.cam.pos[1]; cam_o.z = sx.cam.pos[2];
    kern<<<blocks, FAST_BLOCK, smem, c.stream>>>(sc, sx.nodes, sx.ref_id, sh, w, wh, bounce, q, cam_o, w.cam_origin, seam);
}
void mfx_h_extend(const LaunchCfg &c, const SceneF &sc, const SceneX &sx, const SceneH &sh, const WaveF &w, const WaveH &wh, int bounce, HybQuery q, int seam)
{
    cudaMemsetAsync(wh.fix_n, 0, sizeof(int), c.stream);
    switch (c.hyb_variant) {        // tuning knob (MFX_HYB_VARIANT, tools/hyb_sweep.py); <refill, leaf vote, node steps, blocks/SM>
    case 1: launch_h_trace<16, 10, 2, 4>(c, sc, sx, sh, w, wh, bounce, q, seam); break;
    case 2: launch_h_trace<16, 10, 2, 3>(c, sc, sx, sh, w, wh, bounce, q, seam); break;
    case 3: launch_h_trace<16, 16, 2, 4>(c, sc, sx, sh, w, wh, bounce, q, seam); break;
    case 4: launch_h_trace<16, 10, 2, 6>(c, sc, sx, sh, w, wh, bounce, q, seam); break;
    case 5: launch_h_trace<16, 10, 1, 5>(c, sc, sx, sh, w, wh, bounce, q, seam); break;
    case 6: launch_h_trace<8, 10, 2, 5>(c, sc, sx, sh, w, wh, bounce, q, seam); break;
    case 7: launch_h_trace<24, 16, 2, 5>(c, sc, sx, sh, w, wh, bounce, q, seam); break;     // (7..10: thresholds for the coherent warps the path-id order gives)
    case 8: launch_h_trace<16, 16, 2, 5>(c, sc, sx, sh, w, wh, bounce, q, seam); break;
    case 9: launch_h_trace<24, 10, 2, 5>(c, sc, sx, sh, w, wh, bounce, q, seam); break;
    case 10: launch_h_trace<28, 20, 2, 5>(c, sc, sx, sh, w, wh, bounce, q, seam); break;
    default: launch_h_trace<16, 10, 2, 5>(c, sc, sx, sh, w, wh, bounce, q, seam); break;
    }
    k_h_fixup<<<c.blocks * 4, 128, 0, c.stream>>>(sx, sh, w, wh, bounce, q, w.cam_origin, seam);
}
void mfx_h_extend_x(const LaunchCfg &c, const SceneF &sc, const SceneX &sx, const SceneH &sh, const WaveX &wx, const WaveF &w, const WaveH &wh, int bounce, HybQuery q)
{
    k_h_gather_x<<<persistent_blocks(k_h_gather_x, 256, c.blocks), 256, 0, c.stream>>>(wx, w, wh, bounce);
    mfx_h_extend(c, sc, sx, sh, w, wh, 0, q, 1);
    k_h_scatter_x<<<persistent_blocks(k_h_scatter_x, 256, c.blocks), 256, 0, c.stream>>>(wx, wh, bounce);
}
void mfx_h_shadow_x(const LaunchCfg &c, const SceneX &sx, const SceneF &ref_layout, const SceneH &sh, const WaveX &wx, int bounce)
{
    const float3 lo = make_float3(ref_layout.root_min[0], ref_layout.root_min[1], ref_layout.root_min[2]);
    const float3 hi = make_float3(ref_layout.root_max[0], ref_layout.root_max[1], ref_layout.root_max[2]);
    k_h_shadow_x<<<persistent_blocks(k_h_shadow_x, 128, c.blocks), 128, 0, c.stream>>>(sx, ref_layout.pairs, lo, hi, ref_layout.root_meta, wx, bounce,
                                                                                       sh.max_abs, sh.pad_factor);
}
void mfx_h_guard(cudaStream_t st, const WaveF &w, unsigned long long *totals) { k_h_guard<<<1, 1, 0, st>>>(w.counts, totals); }
void mfx_h_seam_read(const LaunchCfg &c, const SceneX &sx, const WaveH &wh, int n, long long first, int *prim, int *sub, double *t)
{
    k_h_seam_read<<<persistent_blocks(k_h_seam_read, 256, c.blocks), 256, 0, c.stream>>>(sx, wh, n, first, prim, sub, t);
}
